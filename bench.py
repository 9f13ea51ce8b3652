#!/usr/bin/env python
"""Benchmark of the per-marker quantification hot path (BASELINE.json metric: ROI-pixels/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config c1..c5] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Default workload (config.workload): BASELINE config 3, "chip time series" -- per rank 50
timepoints x 4 channels of 4x4 tiles of 2048^2 uint16 (26.8 GB), overlap 102, flat-field correction
on, 1792 buttons (56x32), roi_length 72, per-marker fg/bg counts, sums, means AND medians.  One
step = the whole hot path over that stack: flat-field max pass -> all-reduce(MAX) -> flat-field
apply fused with stitch -> ROI gather fused with all the masked reductions.  Weak scaling: every
rank owns its own block of 50 timepoints; the only collectives are the 2 x float64 MAX all-reduce
and the gather of the per-marker summaries.  `--config c1|c2|c4|c5` runs the other BASELINE
configurations the same way (c4 has no markers: tile pixels per second).

value    = ROI pixels of all ranks / (max-over-ranks device time), inputs resident in HBM.
e2e      = the same metric through the REGISTERED COMPONENTS (`magnify_b200.components`: the
           factories `install()` puts into magnify's registry, chained like Pipeline.__call__) from
           pinned HOST tiles: H2D of the tiles and D2H of image + roi + summaries inside the timed
           region; `e2e_roi_only` is the same without the stitched image coming back (the
           reference's `drop(roi_only=True)`, postprocess.py:6-17); `pcie` is a bare pinned-copy
           probe in the same process layout, the denominator of `frac_of_pcie`.
roofline = the slowest kernel of the step: algorithmic bytes / CUDA-event time against the
           measured copy bandwidth; `stages` lists every stage the same way.
strong_scaling = the named shapes split over the ranks of this run: config 3 (50 timepoints / N)
           and config 5 (100 timepoints / N, in HBM-sized chunks).
parity   = after the timed region: sampled timepoints of the full-size result against torch
           float64 eager arithmetic and plain slicing.
cpu_baseline = the NumPy oracle (the reference's arithmetic, in RAM, no dask/zarr spill) on a
           bounded sample, timed on this box's host cores (rank 0, N=1 only).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "roi_pixels_per_sec"
UNIT = "ROI-px/s"

# BASELINE.json configs (SURVEY.md section 8: C1..C5).  `t` = timepoints per rank of the weak-scaling run.
CONFIGS = {
    "c1": dict(kind="beads", c=9, t=1, r=1, cc=1, h=2048, w=2048, overlap=0, n_beads=300, min_radius=10, max_radius=25,
               roi_length=100, flatfield=True,
               workload="C1 mg.mrbles-sized image: 9 channels of one 2048^2 tile, 300 beads, roi_length 100"),
    "c2": dict(kind="chip", c=2, t=1, r=4, cc=4, h=2048, w=2048, overlap=102, rows=56, cols=32, row_dist=126.1,
               col_dist=232.9, roi_length=72, chamber_radius=30, max_button_radius=15, flatfield=False,
               workload="C2 chip pipeline: 1 timepoint x 2 channels, 4x4 tiles of 2048^2, 56x32 buttons, no flat-field "
                        "(the chip pipe has none, registry.py:243-269)"),
    "c3": dict(kind="chip", c=4, t=50, r=4, cc=4, h=2048, w=2048, overlap=102, rows=56, cols=32, row_dist=126.1,
               col_dist=232.9, roi_length=72, chamber_radius=30, max_button_radius=15, flatfield=True,
               workload="C3 chip time series: flat-field + stitch + ROI gather + fg/bg masks + masked sums/means/medians"),
    "c4": dict(kind="stitch", c=4, t=20, r=10, cc=10, h=2048, w=2048, overlap=102, flatfield=True,
               workload="C4 stitch + flat-field sweep: 10x10 tiles of 2048^2, 4 channels, 20 timepoints (67 GB)"),
    "c5": dict(kind="beads", c=4, t=10, r=10, cc=10, h=2048, w=2048, overlap=0, n_beads=100000, min_radius=4, max_radius=12,
               roi_length=50, flatfield=True,
               workload="C5 bead screen shard: 20480^2 images (10x10 tiles, overlap 0), 1e5 beads, roi_length 50; "
                        "10 timepoints resident per rank (100 timepoints over 8 GPUs = 12.5, in chunks)"),
}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""

    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def workload_config(name, cfg, n_gpus):
    """The `config` object of the JSON line -- identical for the GPU arm and the reference arm."""
    return {
        "workload": cfg["workload"], "name": name,
        "tiles_per_rank": [cfg["c"], cfg["t"], cfg["r"], cfg["cc"], cfg["h"], cfg["w"]],
        "overlap": cfg["overlap"], "roi_length": cfg.get("roi_length"), "flatfield": cfg["flatfield"],
        "markers": cfg["rows"] * cfg["cols"] if cfg["kind"] == "chip" else cfg.get("n_beads", 0),
        "sharding": f"time x{n_gpus} (each rank its own {cfg['t']} timepoints)",
        "cache": "inputs far exceed the 126 MB L2 at full size; no explicit flush",
        "arithmetic": "uint16 pixels in and out; flat-field in float64 (exact reference rounding); integer sums; exact medians",
    }


# ----------------------------------------------------------------------------------------------
# CPU arm: the oracle restatement of the reference's arithmetic, chunked per tile over a thread
# pool the way dask's threaded scheduler runs the reference's per-tile chunks.
# ----------------------------------------------------------------------------------------------
def cpu_sample(cfg, seed=0):
    """Host-generated bounded sample of the workload: ONE timepoint, all channels."""
    from magnify_b200 import synth

    rng = np.random.default_rng(seed)
    c, r, cc, h, w = cfg["c"], cfg["r"], cfg["cc"], cfg["h"], cfg["w"]
    if cfg["kind"] == "stitch" or cfg.get("n_beads", 0) > 10000:
        c = 1                                       # 100 tiles of one channel = 0.84 GB per pass
    tiles = np.clip(rng.normal(400, 20, (c, 1, r, cc, h, w)), 0, 65535).astype(np.uint16)
    flat, dark = synth.smooth_flat_dark(h, w) if cfg["flatfield"] else (1.0, 0.0)
    kh, kw = h - cfg["overlap"], w - cfg["overlap"]
    out = dict(tiles=tiles, flat=flat, dark=dark)
    if cfg["kind"] == "chip":
        rows, cols = cfg["rows"], cfg["cols"]
        y0 = (r * kh - (rows - 1) * cfg["row_dist"]) / 2
        x0 = (cc * kw - (cols - 1) * cfg["col_dist"]) / 2
        cy = y0 + np.arange(rows)[:, None] * cfg["row_dist"] + rng.uniform(-2, 2, (rows, cols))
        cx = x0 + np.arange(cols)[None, :] * cfg["col_dist"] + rng.uniform(-2, 2, (rows, cols))
        m = rows * cols
        out.update(x=cx.reshape(m, 1), y=cy.reshape(m, 1),
                   rad=(10 + (np.add.outer(np.arange(rows), np.arange(cols)) % 6)).reshape(m, 1).astype(np.int32))
    elif cfg["kind"] == "beads":
        n = min(cfg["n_beads"], 5000)               # the label raster of the port is a Python-speed loop per bead
        out["beads"] = np.stack([rng.integers(0, r * kh, n), rng.integers(0, cc * kw, n),
                                 rng.integers(cfg["min_radius"], cfg["max_radius"] + 1, n)], 1).astype(np.float64)
    return out


def cpu_hot_path(cfg, s, threads):
    from concurrent.futures import ThreadPoolExecutor

    from oracle import flatfield as o_ff, reduce as o_red, rois as o_rois, stitch as o_st

    tiles = s["tiles"]
    c, t, r, cc, h, w = tiles.shape
    idx = [(a, b, i, j) for a in range(c) for b in range(t) for i in range(r) for j in range(cc)]
    with ThreadPoolExecutor(max_workers=threads) as pool:
        if cfg["flatfield"]:
            maxima = list(pool.map(lambda k: o_ff.flatfield_maxima(tiles[k], s["flat"], s["dark"]), idx))
            m1 = max(m[0] for m in maxima)
            m2 = max(m[1] for m in maxima)
            out = np.empty_like(tiles)

            def apply(k):
                out[k] = o_ff.flatfield_correct(tiles[k], s["flat"], s["dark"], maxima=(m1, m2))

            list(pool.map(apply, idx))
        else:
            out = tiles
        image = o_st.stitch(out, cfg["overlap"])
        if cfg["kind"] == "stitch":
            return tiles.size
        length = cfg["roi_length"]
        if cfg["kind"] == "chip":
            x, y = s["x"], s["y"]
            fg, bg = o_rois.chip_masks(x[:, 0], y[:, 0], s["rad"][:, 0], length, cfg["chamber_radius"],
                                       cfg["max_button_radius"], image.shape[-1], image.shape[-2])
        else:
            beads = s["beads"]
            x, y = beads[:, 1:2], beads[:, 0:1]
            _, fg, bg = o_rois.bead_masks(beads, image.shape[-2], image.shape[-1], length)
        roi = o_rois.gather_rois(image, x, y, length)
        fgt, bgt = np.repeat(fg[:, None], t, 1), np.repeat(bg[:, None], t, 1)
        parts = [p for p in np.array_split(np.arange(roi.shape[0]), max(1, threads)) if len(p)]
        list(pool.map(lambda p: o_red.masked_stats(roi[p], fgt[p], bgt[p]), parts))
        return roi.size


def time_cpu(cfg, steps, warmup, threads):
    s = cpu_sample(cfg)
    times, px = [], 0
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        px = cpu_hot_path(cfg, s, threads)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    total = sum(times)
    markers = len(s["x"]) if "x" in s else (len(s["beads"]) if "beads" in s else 0)
    sample = (f"1 timepoint x {s['tiles'].shape[0]} channel(s) of the {cfg['r']}x{cfg['cc']} tile grid of {cfg['h']}x{cfg['w']}"
              + (f", {markers} markers of {cfg['roi_length']}^2" if markers else "") + ", data in RAM, NumPy oracle over a "
              f"{threads}-thread pool")
    return px * len(times) / total, total / len(times), sample


def run_reference_arm(args, name, cfg):
    """--impl reference: the reference's CPU arithmetic (oracle port; the reference itself is
    pure Python that cannot be imported on the GPU box -- xarray/dask/zarr are absent) on the host cores."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    threads = os.cpu_count() or 1
    value, sec_per_step, sample = time_cpu(cfg, args.steps, args.warmup, threads)
    unit = UNIT if cfg["kind"] != "stitch" else "tile-px/s"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": unit, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec_per_step * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(name, cfg, args.gpus),
        "cpu_baseline": {"value": value, "unit": unit, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def build_case(cfg, seed, dev, group, timepoints=None):
    """Synthetic stack + plan with markers set (device-resident)."""
    from magnify_b200 import pipeline, synth

    t = cfg["t"] if timepoints is None else timepoints
    if cfg["kind"] == "chip":
        keys = ("c", "r", "cc", "h", "w", "overlap", "rows", "cols", "row_dist", "col_dist", "roi_length",
                "chamber_radius", "max_button_radius")
        case = synth.chip_case(**{k: cfg[k] for k in keys}, t=t, seed=seed, device=dev)
    else:
        case = synth.bead_case(c=cfg["c"], t=t, r=cfg["r"], cc=cfg["cc"], h=cfg["h"], w=cfg["w"], overlap=cfg["overlap"],
                               n_beads=max(cfg.get("n_beads", 0), 1), min_radius=cfg.get("min_radius", 4),
                               max_radius=cfg.get("max_radius", 12), roi_length=cfg.get("roi_length") or 50, seed=seed,
                               device=dev)
    flat, dark = (case.flat, case.dark) if cfg["flatfield"] else (1.0, 0.0)
    plan = pipeline.QuantifyPlan(case.tiles.shape, case.overlap, case.roi_length, flat, dark, device=dev, group=group)
    if cfg["kind"] == "chip":
        plan.set_chip_markers(case.x, case.y, case.fg_radius, case.chamber_radius, case.max_button_radius)
    elif cfg["kind"] == "beads":
        plan.set_bead_markers(case.beads)
    return case, plan


def stage_bytes_table(cfg, tile_px, roi_px, phi):
    table = {"flatfield_max": 2.0 * tile_px,
             "flatfield_stitch": ((2.0 + 2.0 * phi) if cfg["flatfield"] else 4.0 * phi) * tile_px}
    if cfg["kind"] != "stitch":
        table["roi_gather_stats"] = 4.0 * roi_px
    return table


KERNEL_OF = {
    "flatfield_max": "ff_tilemax_u16_kernel (+ ff_maxima_kernel)",
    "flatfield_stitch": "stitch_u16_kernel (flat-field apply fused with stitch when flat-field is on; timed together with "
                        "the 0.03 ms coefficient-table kernel)",
    "roi_gather_stats": "roi_gather_lists_kernel (TMA-staged ROI gather fused with counts, sums, means and medians)",
}


def run_b200_arm(args, name, cfg):
    import torch
    import torch.distributed as dist

    from magnify_b200 import _lib, numa, ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device; magnify_b200 has no CPU path")
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    if world > 1:
        numa.bind_to_gpu_numa(local_rank)
    group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
    lib = _lib.load()
    peak, peak_src = load_peaks()

    def barrier():
        if world > 1:
            dist.barrier(group=group)
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms: float) -> float:
        v = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(v, op=dist.ReduceOp.MAX, group=group)
        return float(v.item())

    case, plan = build_case(cfg, rank, dev, group)
    c, t = cfg["c"], cfg["t"]
    has_markers = cfg["kind"] != "stitch"
    m = plan.boxes.shape[0] if has_markers else 0
    length = plan.roi_length
    image_out = ops.alloc_image(plan.image_shape, torch.uint16, dev)
    roi_out = torch.empty((m, c, t, length, length), dtype=torch.uint16, device=dev) if has_markers else None
    stats_out = torch.empty((m, c, t, ops.NSTATS), dtype=torch.float64, device=dev) if has_markers else None
    gathered = None
    if world > 1 and has_markers:
        gathered = torch.empty((world,) + tuple(stats_out.shape), dtype=torch.float64, device=dev)
    symm = None
    if world > 1 and has_markers and not args.no_fused_gather:
        try:  # summaries all-gathered by the gather kernel itself over NVLink peer memory
            from magnify_b200.dist import SymmetricSummaries

            symm = SymmetricSummaries(stats_out.shape, dev, group)
        except Exception as exc:
            print(f"[bench] symmetric memory unavailable ({exc!r}); using NCCL all_gather", file=sys.stderr)
            symm = None
    if symm is not None:   # the peer stores only exist in the fused kernel; masks beyond its lists take the local path
        plan.run_device(case.tiles, want_roi=False, image_out=image_out, stats_out=stats_out)
        if not ops.last_gather_fused:
            print("[bench] masks exceed the fused gather's value lists; summaries go through NCCL all_gather", file=sys.stderr)
            symm = None
    roi_px_rank = m * c * t * length * length
    tile_px_rank = case.tiles.numel()
    phi = (plan.image_shape[-1] * plan.image_shape[-2]) / (cfg["r"] * cfg["cc"] * cfg["h"] * cfg["w"])
    unit_px_rank = roi_px_rank if has_markers else tile_px_rank
    unit = UNIT if has_markers else "tile-px/s"

    def step(record=None):
        if not has_markers:
            stream = torch.cuda.current_stream(dev)
            a, mid, b = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            a.record(stream)
            maxima = None
            if not plan.ff.identity:
                maxima = ops.flatfield_maxima(case.tiles, plan.ff)
                if world > 1:
                    dist.all_reduce(maxima, op=dist.ReduceOp.MAX, group=group)
            mid.record(stream)
            ops.flatfield_stitch(case.tiles, overlap=plan.overlap, plan=plan.ff, maxima=maxima, out=image_out)
            b.record(stream)
            if record is not None:
                if not plan.ff.identity:
                    record.append(("flatfield_max", a, mid))
                record.append(("flatfield_stitch", mid, b))
            return
        if symm is not None:
            plan.run_device(case.tiles, want_roi=True, image_out=image_out, roi_out=roi_out, record=record,
                            peer_stats=symm.peer_blocks)
            symm.barrier()
            return
        plan.run_device(case.tiles, want_roi=True, image_out=image_out, roi_out=roi_out, stats_out=stats_out, record=record)
        if world > 1:
            dist.all_gather_into_tensor(gathered, stats_out, group=group)

    warmup = max(args.warmup, 3)
    for _ in range(warmup):
        step()
    barrier()
    if symm is not None:   # the fused gather must equal the NCCL all-gather of the same summaries
        plan.run_device(case.tiles, want_roi=False, image_out=image_out, stats_out=stats_out)
        dist.all_gather_into_tensor(gathered, stats_out, group=group)
        torch.cuda.synchronize(dev)
        same = torch.equal(torch.nan_to_num(gathered, nan=-1.0), torch.nan_to_num(symm.gathered, nan=-1.0))
        if not same:
            raise RuntimeError("fused peer-store gather of the summaries differs from the NCCL all_gather")
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    launches0 = lib.mgb_launch_count()
    records = []
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    start.record()
    for _ in range(args.steps):
        rec = []
        step(rec)
        records.append(rec)
    end.record()
    barrier()
    launches = lib.mgb_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        outputs = {"image": image_out}
        if has_markers:
            outputs.update(roi=roi_out, stats=symm.gathered[rank] if symm is not None else stats_out)
        dump_outputs(args.dump_outputs, outputs)
    elapsed_s = max_over_ranks(start.elapsed_time(end)) / 1e3
    value = unit_px_rank * world * args.steps / elapsed_s

    # per-stage device times (this rank), averaged over the timed steps
    stage_ms = {}
    for rec in records:
        for sname, a, b in rec:
            stage_ms.setdefault(sname, []).append(a.elapsed_time(b))
    stage_ms = {k: sum(v) / len(v) for k, v in stage_ms.items()}
    sbytes = stage_bytes_table(cfg, tile_px_rank, roi_px_rank, phi)
    stages = {}
    for sname, ms in stage_ms.items():
        entry = {"ms": ms}
        if sname in sbytes and ms > 0:
            gbs = sbytes[sname] / (ms * 1e-3) / 1e9
            entry.update({"algorithmic_GB": sbytes[sname] / 1e9, "GB/s": gbs, "frac_of_peak": gbs / peak})
        stages[sname] = entry
    timed = {k: v for k, v in stage_ms.items() if k in sbytes}
    dom = max(timed, key=timed.get) if timed else None
    traffic, traffic_note = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")   # dram bytes per launch from ncu --set full
    if dom and os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        entry = tj.get(f"{name}:{dom}:T={cfg['t']}")
        if isinstance(entry, dict):
            traffic, traffic_note = entry.get("dram_bytes"), f"ncu --set full at commit {entry.get('commit')}"
    kernel_of = dict(KERNEL_OF)
    if has_markers and not ops.last_gather_fused:   # masks too large for the in-kernel value lists (config 1: L = 100)
        kernel_of["roi_gather_stats"] = ("roi_gather_tma_kernel (TMA-staged ROI gather fused with counts / sums / means) + "
                                         "2 x roi_median_kernel (stand-alone exact medians): masks beyond the fused kernel's "
                                         "1024 fg / 2560 bg values per marker")
    achieved = stages[dom]["GB/s"] if dom else None
    step_bytes = sum(sbytes[k] for k in timed)
    roofline = {
        "bound": "hbm", "kernel": kernel_of.get(dom), "stage": dom,
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
        "traffic": traffic, "traffic_source": traffic_note, "peak_source": peak_src,
        "algorithmic_bytes_per_launch": sbytes.get(dom), "avg_launch_ms": stage_ms.get(dom),
        "stages": stages,
        "step": {"algorithmic_GB": step_bytes / 1e9, "GB/s": step_bytes / (elapsed_s / args.steps) / 1e9,
                 "frac_of_peak": step_bytes / (elapsed_s / args.steps) / 1e9 / peak},
    }

    # ---- sampled full-size parity of what was just timed (outside the timed region)
    parity = None
    if not args.no_parity:
        try:
            got_stats = None if not has_markers else (symm.gathered[rank] if symm is not None else stats_out)
            parity = sampled_parity(case, plan, image_out, roi_out, got_stats, group)
        except Exception as exc:
            parity = {"ok": False, "error": repr(exc)[:300]}

    host_case = dict(x=getattr(case, "x", None), y=getattr(case, "y", None), fg_radius=getattr(case, "fg_radius", None),
                     beads=getattr(case, "beads", None), flat=case.flat, dark=case.dark)
    tiles_dev = [case.tiles]                # handed over (and released) inside measure_e2e
    del image_out, roi_out, stats_out, gathered, plan, case
    torch.cuda.empty_cache()

    # ---- the host legs: link probe, then the registered components from pinned host memory
    e2e = e2e_roi = pcie = None
    try:
        pcie = pcie_probe(dev, world, barrier, max_over_ranks)
    except Exception as exc:
        pcie = {"error": repr(exc)[:300]}
    try:
        e2e, e2e_roi = measure_e2e(args, cfg, host_case, tiles_dev, dev, world, group, barrier, max_over_ranks, pcie)
    except Exception as exc:  # keep the device numbers even if the host leg cannot allocate
        e2e = {"value": None, "unit": unit, "error": repr(exc)[:300]}
    tiles_dev.clear()
    torch.cuda.empty_cache()

    # ---- strong scaling on the named shapes (this run's N)
    strong = None
    if not args.no_strong and name == "c3":
        try:
            strong = strong_scaling(args, dev, rank, world, group, barrier, max_over_ranks,
                                    None if world > 1 else (elapsed_s / args.steps))
        except Exception as exc:
            strong = {"error": repr(exc)[:300]}

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v, sec, sample = time_cpu(cfg, steps=3, warmup=1, threads=threads)
        cpu_baseline = {"value": v, "unit": unit, "cores": threads, "kind": "port",
                        "sample": f"{sample}; 3 timed passes of {sec:.2f} s (~{4 * sec * threads:.0f} core-seconds)"}
    elif rank == 0:
        cpu_baseline = {"value": None, "note": "measured on rank 0 at N=1 only (bench.py --gpus 1, or --impl reference)"}
    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": elapsed_s * 1e3 / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u16", "data": "synthetic",
            "config": workload_config(name, cfg, world),
            "summary_gather": ("fused peer stores over NVLink (symmetric memory)" if symm is not None
                               else ("nccl all_gather" if world > 1 else "single rank")),
            "clocks": clocks, "e2e": e2e, "e2e_roi_only": e2e_roi, "pcie": pcie, "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": cpu_baseline, "parity": parity, "strong_scaling": strong,
        }
    if world > 1:
        dist.barrier(group=group)
        dist.destroy_process_group()
    return line


DUMP_MAX_ELEMENTS = 1 << 20


def dump_outputs(directory, outputs):
    """Write the arrays of the last timed step as DIR/<name>.npy (uint16 -> float32, float64 kept)
    so that two builds can be compared output for output.  An array of more than
    DUMP_MAX_ELEMENTS elements is replaced by a sample at fixed, seeded flat (C-order) positions,
    written beside it as DIR/<name>_index.npy (float64); every file together stays under 64 MB."""
    import torch

    os.makedirs(directory, exist_ok=True)
    for seed, (name, tensor) in enumerate(outputs.items()):
        dtype = np.float64 if tensor.dtype == torch.float64 else np.float32
        # CUDA indexing has no uint16 kernel: gather the same bits as int16 and reinterpret on the host
        unsigned16 = tensor.dtype == torch.uint16
        src = tensor.view(torch.int16) if unsigned16 else tensor
        n = tensor.numel()
        if n <= DUMP_MAX_ELEMENTS:
            values = src.cpu().numpy()
        else:
            index = np.unique(np.random.default_rng(seed).integers(0, n, DUMP_MAX_ELEMENTS, dtype=np.int64))
            coords = tuple(torch.from_numpy(a).to(tensor.device) for a in np.unravel_index(index, tuple(tensor.shape)))
            values = src[coords].cpu().numpy()
            np.save(os.path.join(directory, f"{name}_index.npy"), index.astype(np.float64))
        if unsigned16:
            values = values.view(np.uint16)
        np.save(os.path.join(directory, f"{name}.npy"), values.astype(dtype))


def sampled_parity(case, plan, image, roi, stats, group=None):
    """Timepoints {0, T/2, T-1} of the full-size result against torch float64 eager arithmetic
    (flat-field: the reference's operation order; IEEE float64 on the GPU is bit-identical to
    NumPy's), plain slicing (stitch, crops) and torch sorts / sums (summaries of 64 sampled markers)."""
    import torch

    c, t, r, cc, h, w = case.tiles.shape
    ov = case.overlap
    clip, rem = ov // 2, ov % 2
    times = sorted({0, t // 2, t - 1})
    checked = {"image_planes": 0, "crops": 0, "summaries": 0}
    m1 = m2 = None
    if not plan.ff.identity:
        flat, dark = plan.ff.flat, plan.ff.dark               # (K,H,W) float64
        m1 = torch.zeros((), dtype=torch.float64, device=image.device)
        m2 = torch.zeros((), dtype=torch.float64, device=image.device)
        for ci in range(c):
            k = ci if flat.shape[0] > 1 else 0
            for ti in range(t):
                x = (case.tiles[ci, ti].to(torch.float64) - dark[k]).clamp_(min=0)
                m1 = torch.maximum(m1, x.max())
                m2 = torch.maximum(m2, (x / flat[k]).max())
        if group is not None:          # both maxima are global over every rank's tiles (preprocess.py:84,86)
            import torch.distributed as dist

            both = torch.stack([m1, m2])
            dist.all_reduce(both, op=dist.ReduceOp.MAX, group=group)
            m1, m2 = both[0], both[1]
        if not torch.equal(torch.stack([m1, m2]), plan.ff.maxima):
            return {"ok": False, "what": "flat-field maxima differ from torch float64"}
    for ti in times:
        for ci in range(c):
            tiles = case.tiles[ci, ti]
            if not plan.ff.identity:
                k = ci if plan.ff.flat.shape[0] > 1 else 0
                x = (tiles.to(torch.float64) - plan.ff.dark[k]).clamp_(min=0) / plan.ff.flat[k]
                x = (x * m1) / m2
                tiles = x.to(torch.int32).to(torch.uint16)          # truncation, values are in [0, M]
            kept = tiles[..., clip:h - clip - rem, clip:w - clip - rem]
            want = kept.permute(0, 2, 1, 3).reshape(r * (h - ov), cc * (w - ov))
            if not torch.equal(image[ci, ti].contiguous().view(torch.int16), want.contiguous().view(torch.int16)):
                return {"ok": False, "what": f"image[{ci},{ti}] differs from torch float64 + slicing"}
            checked["image_planes"] += 1
    if roi is not None and roi.shape[0] > 0:
        m = roi.shape[0]
        length = plan.roi_length
        sample = sorted(set(torch.linspace(0, m - 1, min(m, 64)).long().tolist()))
        boxes = plan.boxes.cpu()
        mask_t = plan.mask_t.cpu().tolist()
        for mi in sample:
            for ti in times:
                top, left = int(boxes[mi, ti, 0]), int(boxes[mi, ti, 1])
                want = image[:, ti, top:top + length, left:left + length].contiguous()
                if not torch.equal(roi[mi, :, ti].contiguous().view(torch.int16), want.view(torch.int16)):
                    return {"ok": False, "what": f"roi[{mi},:,{ti}] differs from image slicing"}
                checked["crops"] += c
                for col, mask in ((0, plan.fg), (1, plan.bg)):
                    sel = mask[mi, mask_t[ti]].bool()
                    n = int(sel.sum())
                    for ci in range(c):
                        vals = want[ci].to(torch.int32)[sel].to(torch.float64)
                        got = stats[mi, ci, ti]
                        exp_sum = float(vals.sum()) if n else 0.0
                        ok = float(got[col]) == n and float(got[2 + col]) == exp_sum
                        if n:
                            srt = torch.sort(vals).values
                            med = 0.5 * (float(srt[(n - 1) // 2]) + float(srt[n // 2]))
                            mean = exp_sum / n
                            ok = ok and float(got[6 + col]) == med and abs(float(got[4 + col]) - mean) <= 1e-12 * max(1.0, mean)
                        else:
                            ok = ok and bool(torch.isnan(got[4 + col])) and bool(torch.isnan(got[6 + col]))
                        if not ok:
                            return {"ok": False, "what": f"summaries[{mi},{ci},{ti}] ({'fg' if col == 0 else 'bg'}) differ"}
                        checked["summaries"] += 1
    return {"ok": True, "timepoints": times, **checked,
            "against": "torch float64 eager flat-field + slicing + torch sort/sum, on the tensors the timed steps produced"}


def strong_scaling(args, dev, rank, world, group, barrier, max_over_ranks, c3_full_step_s):
    """Config 3 (50 timepoints) and config 5 (100 timepoints) SPLIT over the ranks of this run.
    value = ROI pixels of the whole problem / max-over-ranks device time of the shards."""
    import torch

    from magnify_b200 import dist as mdist

    out = {"n_gpus": world}
    # ---- C3: 50 timepoints / N
    cfg = CONFIGS["c3"]
    total_t = 50
    lo, hi = mdist.shard_timepoints(total_t, rank, world) if world > 1 else (0, total_t)
    roi_px_total = cfg["rows"] * cfg["cols"] * cfg["c"] * total_t * cfg["roi_length"] ** 2
    if world == 1 and c3_full_step_s is not None:
        out["c3"] = {"timepoints_per_rank": total_t, "ms": c3_full_step_s * 1e3, "value": roi_px_total / c3_full_step_s,
                     "note": "N=1: the main measurement"}
    else:
        case, plan = build_case(cfg, 100 + rank, dev, group, timepoints=hi - lo)
        res = time_plan(plan, case, dev, barrier, steps=max(3, args.steps))
        ms = max_over_ranks(res["ms"])
        out["c3"] = {"timepoints_per_rank": hi - lo, "ms": ms, "value": roi_px_total / (ms * 1e-3),
                     "stages_ms": res["stages"]}
        del case, plan
        torch.cuda.empty_cache()
    # ---- C5: 100 timepoints / N, in chunks that fit HBM; one synthetic tile block stands for every
    # chunk (pixel values do not change the work; the medians see the same noise statistics)
    cfg = CONFIGS["c5"]
    total_t = 100
    lo, hi = mdist.shard_timepoints(total_t, rank, world) if world > 1 else (0, total_t)
    mine = hi - lo
    chunk_t = min(mine, 10)
    case, plan = build_case(cfg, 200 + rank, dev, group, timepoints=chunk_t)
    roi_px_total = cfg["n_beads"] * cfg["c"] * total_t * cfg["roi_length"] ** 2
    res = time_plan(plan, case, dev, barrier, steps=3)
    full_chunks, tail = divmod(mine, chunk_t)
    ms_rank = res["ms"] * full_chunks
    tail_ms = None
    del case, plan
    torch.cuda.empty_cache()
    if tail:
        case_t, plan_t = build_case(cfg, 200 + rank, dev, group, timepoints=tail)
        tail_ms = time_plan(plan_t, case_t, dev, barrier, steps=3)["ms"]
        ms_rank += tail_ms
        del case_t, plan_t
        torch.cuda.empty_cache()
    ms = max_over_ranks(ms_rank)
    out["c5"] = {"timepoints_per_rank": mine, "chunk_timepoints": chunk_t, "chunks": full_chunks + (1 if tail else 0),
                 "ms": ms, "value": roi_px_total / (ms * 1e-3), "chunk_ms": res["ms"], "tail_chunk_ms": tail_ms,
                 "stages_ms_per_chunk": res["stages"],
                 "note": "device-resident chunks of <= 10 timepoints (34 GB of tiles + 34 GB of images + 20 GB of crops); "
                         "per-rank time = measured chunk time x chunks of the shard (identical work per chunk)"}
    return out


def time_plan(plan, case, dev, barrier, steps=3):
    import torch

    from magnify_b200 import ops

    c, t = case.tiles.shape[:2]
    m, length = plan.boxes.shape[0], plan.roi_length
    image = ops.alloc_image(plan.image_shape, torch.uint16, dev)
    roi = torch.empty((m, c, t, length, length), dtype=torch.uint16, device=dev)
    stats = torch.empty((m, c, t, ops.NSTATS), dtype=torch.float64, device=dev)
    for _ in range(3):
        plan.run_device(case.tiles, image_out=image, roi_out=roi, stats_out=stats)
    barrier()
    recs = []
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        rec = []
        plan.run_device(case.tiles, image_out=image, roi_out=roi, stats_out=stats, record=rec)
        recs.append(rec)
    b.record()
    barrier()
    stages = {}
    for rec in recs:
        for sname, x, y in rec:
            stages.setdefault(sname, []).append(x.elapsed_time(y))
    return {"ms": a.elapsed_time(b) / steps, "stages": {k: sum(v) / len(v) for k, v in stages.items()}}


def pcie_probe(dev, world, barrier, max_over_ranks, nbytes=1 << 30):
    """Bare pinned cudaMemcpyAsync bandwidth in this process layout: host->device alone,
    device->host alone, both at once (two streams) -- the ceiling the staged pipeline can reach."""
    import torch

    h_in = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    h_out = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    d_in = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    d_out = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def run(up, down, reps=4):
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            if up:
                with torch.cuda.stream(s1):
                    d_in.copy_(h_in, non_blocking=True)
            if down:
                with torch.cuda.stream(s2):
                    h_out.copy_(d_out, non_blocking=True)
        s1.synchronize()
        s2.synchronize()
        sec = max_over_ranks((time.perf_counter() - t0) * 1e3) / 1e3
        barrier()
        return reps * nbytes / sec / 1e9

    run(True, True, 1)
    h2d, d2h, both = run(True, False), run(False, True), run(True, True)
    return {"h2d_GBps_per_gpu": h2d, "d2h_GBps_per_gpu": d2h, "bidirectional_GBps_per_gpu_each_way": both,
            "bidirectional_GBps_per_gpu_total": 2 * both, "bytes_per_copy": nbytes, "ranks_copying_at_once": world,
            "box_total_GBps_bidirectional": 2 * both * world,
            "how": "pinned host <-> device cudaMemcpyAsync of 1 GiB blocks, 4 repetitions, all ranks at the same time"}


def measure_e2e(args, cfg, hc, tiles_dev, dev, world, group, barrier, max_over_ranks, pcie):
    """The hot path through the registered components from pinned host tiles, assays back to back."""
    import psutil
    import torch
    import torch.distributed as dist

    from magnify_b200 import components, devarray
    from magnify_b200.dataset import Dataset

    c, t = cfg["c"], cfg["t"]
    kind = cfg["kind"]
    length = cfg.get("roi_length") or 0
    him, wim = cfg["r"] * (cfg["h"] - cfg["overlap"]), cfg["cc"] * (cfg["w"] - cfg["overlap"])
    m = (cfg["rows"] * cfg["cols"]) if kind == "chip" else (len(hc["beads"]) if kind == "beads" else 0)
    per_t_in = c * cfg["r"] * cfg["cc"] * cfg["h"] * cfg["w"] * 2
    per_t_out = (him * wim * c + m * c * length * length) * 2 + m * c * 64
    avail = psutil.virtual_memory().available
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    # pinned: the input stack once, the outputs of two assays in flight (rounded up by the allocator)
    t_e2e = int(min(t, max(1, (0.6 * avail / local_world) // (per_t_in + 3 * per_t_out))))
    # device: tiles + outputs of two assays in flight must fit without allocator retries (a retry frees
    # cached blocks with a device synchronise, which breaks the upload/download overlap)
    hbm = torch.cuda.get_device_properties(dev).total_memory
    t_e2e = int(min(t_e2e, max(1, (0.8 * hbm) // (2 * (per_t_in + per_t_out)))))
    if args.e2e_timepoints:
        t_e2e = min(t, args.e2e_timepoints)
    if world > 1:  # every rank must agree on the shape of the problem
        tt = torch.tensor([t_e2e], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MIN, group=group)
        t_e2e = int(tt.item())
    shape = (c, t_e2e) + tuple(tiles_dev[0].shape[2:])
    tiles_host = torch.empty(shape, dtype=torch.uint16, pin_memory=True)
    tiles_host.copy_(tiles_dev[0][:, :t_e2e])
    torch.cuda.synchronize(dev)
    tiles_dev.clear()                       # the resident stack of the device-timed leg is not needed any more
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats(dev)
    retries0 = int(torch.cuda.memory_stats(dev).get("num_alloc_retries", 0))
    tiles_np = tiles_host.numpy()

    # the registry `install()` fills, and the chain the reference's builder assembles from it
    class Registry(dict):
        def register(self, name):
            return lambda f: self.__setitem__(name, f) or f

    reg = Registry()
    components.install(registry=reg)
    pipe = []
    if cfg["flatfield"]:
        pipe.append(("flatfield_correct", reg["flatfield_correct"](flatfield=hc["flat"], darkfield=hc["dark"])))
    pipe.append(("stitch", reg["stitch"](overlap=cfg["overlap"])))
    coords = {"channel": (("channel",), np.array([f"ch{k}" for k in range(c)]))}
    if kind == "chip":
        rows, cols = cfg["rows"], cfg["cols"]
        x = hc["x"][:, :t_e2e].reshape(rows, cols, t_e2e)
        y = hc["y"][:, :t_e2e].reshape(rows, cols, t_e2e)
        rad = hc["fg_radius"][:, 0].reshape(rows, cols)
        tag = np.full((rows, cols), "default", dtype="<U200")
        coords.update(tag=(("mark_row", "mark_col"), tag),
                      valid=(("mark_row", "mark_col", "time"), np.ones((rows, cols, t_e2e), dtype=bool)))
        pipe.append(("find_buttons", reg["find_buttons"](
            row_dist=cfg["row_dist"], col_dist=cfg["col_dist"], min_button_diameter=16, max_button_diameter=30,
            chamber_diameter=60, top_chamber=None, left_chamber=None, low_edge_quantile=0.1, high_edge_quantile=0.9,
            num_iter=5000000, min_roundness=0.2, cluster_penalty=50, roi_length=None, progress_bar=False,
            search_timestep=0, search_channel=None, interactive=False,
            centers=lambda xp, ts: (x[..., ts], y[..., ts], rad))))
        pipe.append(("quantify", reg["quantify"]()))
    elif kind == "beads":
        pipe.append(("find_beads", reg["find_beads"](
            min_bead_diameter=2 * cfg["min_radius"], max_bead_diameter=2 * cfg["max_radius"], low_edge_quantile=0.1,
            high_edge_quantile=0.9, num_iter=5000000, min_roundness=0.3, roi_length=length, search_channel=None,
            interactive=False, centers=hc["beads"])))
        pipe.append(("quantify", reg["quantify"]()))

    def run_pipe():
        assay = Dataset({"tile": (components.TILE_DIMS, tiles_np)}, coords=coords)
        for _, component in pipe:            # Pipeline.__call__, pipeline.py:19-22
            assay = component(assay)
        return assay

    def read_back(assay, want_image: bool) -> int:
        """What a caller reads: the crops, the summaries, and (unless roi_only) the stitched image."""
        n = 0
        for name in (["image"] if want_image else []) + (["roi"] if m else []):
            n += np.asarray(assay[name].values).nbytes
        if m:
            n += sum(np.asarray(assay[k].values).nbytes for k in ("fg_mean", "bg_mean", "fg_median", "bg_median", "fg_sum", "bg_sum"))
        return n

    steps = 8 if not args.e2e_timepoints else max(1, min(args.steps, 8))   # assays back to back (the first upload and
    #                                                  the last download overlap with nothing: amortised over the chain)
    results = []
    for want_image in ((True, False) if m else (True,)):
        devarray.PREFETCH_SKIP = () if want_image else ("image",)
        # warm-up in the timed loop's own pattern: two results alive at once, so that the pinned
        # result buffers of BOTH are in the pool before the clock starts (page-locking 28 GB takes seconds)
        prev, d2h = None, 0
        for _ in range(3):
            cur = run_pipe()
            if prev is not None:
                d2h = read_back(prev, want_image)
            prev = cur
        read_back(prev, want_image)
        del prev, cur
        barrier()
        # Wall clock around fully synchronised ends: the region holds every H2D copy, kernel and D2H
        # copy of `steps` assays; the D2H of assay k (copy stream) overlaps the H2D of assay k+1.
        timeline = [] if os.environ.get("MGB_E2E_TIMELINE") else None   # diagnostic: where each stream is per assay
        if timeline is not None:
            streams = devarray.Streams.of(dev)
            watched = (streams.h2d, torch.cuda.current_stream(dev), streams.d2h)
            ev0 = torch.cuda.Event(enable_timing=True)
            ev0.record(watched[1])
            devarray.TRACE = []
        t0 = time.perf_counter()
        prev = None
        for _ in range(steps):
            cur = run_pipe()
            if timeline is not None:
                t_ret = time.perf_counter() - t0
                evs = [torch.cuda.Event(enable_timing=True) for _ in watched]
                for e, st in zip(evs, watched):
                    e.record(st)
            if prev is not None:
                read_back(prev, want_image)
            if timeline is not None:
                timeline.append((t_ret, time.perf_counter() - t0, evs))
            prev = cur
        read_back(prev, want_image)
        torch.cuda.synchronize(dev)
        sec = max_over_ranks((time.perf_counter() - t0) * 1e3) / 1e3
        if timeline is not None:
            for k, (t_ret, t_read, evs) in enumerate(timeline):
                print(f"[e2e timeline image={want_image}] assay {k}: run_pipe returned {1e3 * t_ret:8.1f} ms, previous read "
                      f"{1e3 * t_read:8.1f} ms | h2d done {ev0.elapsed_time(evs[0]):8.1f}  compute done "
                      f"{ev0.elapsed_time(evs[1]):8.1f}  d2h done {ev0.elapsed_time(evs[2]):8.1f} ms", file=sys.stderr)
            for shape, nbytes, began, done in devarray.TRACE:
                if nbytes >= (64 << 20):
                    print(f"[e2e timeline image={want_image}] download {nbytes / 1e9:6.2f} GB {shape}: "
                          f"{ev0.elapsed_time(began):8.1f} -> {ev0.elapsed_time(done):8.1f} ms", file=sys.stderr)
            devarray.TRACE = None
            print(f"[e2e timeline image={want_image}] total {1e3 * sec:.1f} ms", file=sys.stderr)
        del prev, cur
        barrier()
        units = (m * c * t_e2e * length * length) if m else (c * t_e2e * cfg["r"] * cfg["cc"] * cfg["h"] * cfg["w"])
        mem = torch.cuda.memory_stats(dev)
        h2d = tiles_host.numel() * 2
        gbps = (h2d + d2h) * steps / sec / 1e9
        entry = {
            "value": units * world * steps / sec, "unit": UNIT if m else "tile-px/s", "h2d_bytes_per_step": int(h2d),
            "d2h_bytes_per_step": int(d2h), "timepoints": t_e2e, "steps": steps, "ms_per_step": sec * 1e3 / steps,
            "h2d_plus_d2h_GBps_per_gpu": gbps,
            "path": "registered components (" + " -> ".join(n for n, _ in pipe) + ") chained like Pipeline.__call__",
            "outputs_copied_back": ("stitched image + " if want_image else "") + ("roi + summaries" if m else "image"),
            "device_allocator": {"alloc_retries": int(mem.get("num_alloc_retries", 0)) - retries0,
                                 "peak_reserved_GB": mem.get("reserved_bytes.all.peak", 0) / 1e9},
        }
        if pcie and "bidirectional_GBps_per_gpu_each_way" in pcie:
            # the link-bound time of a step that moves h2d and d2h bytes concurrently: no direction faster than
            # alone, both together no faster than the measured bidirectional total
            floor = max(h2d / (pcie["h2d_GBps_per_gpu"] * 1e9), d2h / (pcie["d2h_GBps_per_gpu"] * 1e9),
                        (h2d + d2h) / (pcie["bidirectional_GBps_per_gpu_total"] * 1e9))
            entry["pcie_bound_ms_per_step"] = floor * 1e3
            entry["frac_of_pcie"] = floor / (sec / steps)
        results.append(entry)
    devarray.PREFETCH_SKIP = ()
    return results[0], (results[1] if len(results) > 1 else None)


class StdoutToStderr:
    """Everything written to fd 1 while active goes to stderr (NCCL prints its version banner to
    stdout); the JSON line is printed after restoring, so stdout carries exactly one line."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--timepoints", type=int, default=None, help="timepoints per rank (default: the config's)")
    ap.add_argument("--e2e-timepoints", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--no-fused-gather", action="store_true",
                    help="N>1: gather the summaries with NCCL all_gather instead of peer stores from the kernel")
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS),
                    help="c3 = BASELINE config 3 (default, the metric's workload); c1, c2, c4, c5 = the other configs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the image, crops and summaries of the last step as DIR/<name>.npy "
                         "(large arrays as a fixed, seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    cfg = dict(CONFIGS[args.config])
    if args.timepoints:
        cfg["t"] = args.timepoints
    if args.impl == "reference":
        run_reference_arm(args, args.config, cfg)
    else:
        with StdoutToStderr():
            line = run_b200_arm(args, args.config, cfg)
        if line is not None:
            print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
