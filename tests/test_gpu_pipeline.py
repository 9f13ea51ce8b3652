"""QuantifyPlan / HostStagedRunner end to end against the oracle: several search timesteps with
copy-forward (find.py:143-181), per-channel flat fields, the pinned-host staging loop."""
import numpy as np
import pytest
import torch

from oracle import flatfield as o_ff
from oracle import reduce as o_red
from oracle import rois as o_rois
from oracle import stitch as o_st

pytestmark = pytest.mark.gpu


def oracle_chip(tiles, flat, dark, overlap, x, y, radius, search, length, chamber_r, max_r):
    image = o_st.stitch(o_ff.flatfield_correct(tiles, flat, dark), overlap)
    t = tiles.shape[1]
    src = o_rois.chip_copy_forward(t, search)
    roi = o_rois.gather_rois(image, x, y, length)
    m = x.shape[0]
    fg = np.empty((m, t, length, length), bool)
    bg = np.empty_like(fg)
    searched = sorted(set(src.tolist()))
    for k, ts in enumerate(searched):
        f, b = o_rois.chip_masks(x[:, ts], y[:, ts], radius[:, k], length, chamber_r, max_r, image.shape[-1], image.shape[-2])
        for ti in np.where(src == ts)[0]:
            fg[:, ti], bg[:, ti] = f, b
    return image, roi, fg, bg, o_red.masked_stats(roi, fg, bg)


@pytest.mark.parametrize("search,per_channel", [([0], False), ([1, 3], True)])
def test_chip_plan_matches_oracle(cuda_device, search, per_channel):
    from magnify_b200 import pipeline

    rng = np.random.default_rng(8)
    c, t, r, cc, h, w, ov, length = 2, 5, 2, 4, 128, 128, 22, 40
    tiles = np.clip(rng.normal(3000, 900, (c, t, r, cc, h, w)), 0, 65535).astype(np.uint16)
    flat = 0.7 + 0.6 * rng.random((h, w))
    dark = 95.0 + 10 * rng.random((h, w))
    if per_channel:
        flat = np.stack([flat, flat * 1.2])[:, None, None, None]
        dark = np.stack([dark, dark - 4.0])[:, None, None, None]
    him, wim = r * (h - ov), cc * (w - ov)
    m = 7
    src = o_rois.chip_copy_forward(t, search)
    x_s = rng.uniform(0, wim, (m, t))
    y_s = rng.uniform(0, him, (m, t))
    x, y = x_s[:, src], y_s[:, src]        # centres of non-search timesteps are copied forward
    radius = rng.integers(3, 9, (m, len(set(src.tolist())))).astype(np.int32)
    plan = pipeline.QuantifyPlan(tiles.shape, ov, length, flat, dark, device=cuda_device)
    plan.set_chip_markers(x, y, radius, chamber_radius=16, max_button_radius=9, search_timesteps=search)
    res = plan.run_device(torch.from_numpy(tiles).to(cuda_device))
    image, roi, fg, bg, stats = oracle_chip(tiles, flat, dark, ov, x, y, radius, search, length, 16, 9)
    np.testing.assert_array_equal(res.image.cpu().numpy(), image)
    np.testing.assert_array_equal(res.roi.cpu().numpy(), roi)
    mask_t = res.mask_t.cpu().numpy()
    np.testing.assert_array_equal(res.fg.cpu().numpy().astype(bool)[:, mask_t], fg)
    np.testing.assert_array_equal(res.bg.cpu().numpy().astype(bool)[:, mask_t], bg)
    np.testing.assert_allclose(res.stats.cpu().numpy(), stats, rtol=1e-12, equal_nan=True)


@pytest.mark.parametrize("cc", [4, 3])   # 3 tile columns: stitched width 702 is not a multiple of 8 (padded rows)
def test_host_staged_runner_equals_device_run(cuda_device, cc):
    from magnify_b200 import pipeline, synth

    case = synth.chip_case(c=2, t=3, r=2, cc=cc, h=256, w=256, overlap=22, rows=3, cols=2, row_dist=126.1,
                           col_dist=250.0, seed=2, device=cuda_device)
    plan = pipeline.QuantifyPlan(case.tiles.shape, case.overlap, case.roi_length, case.flat, case.dark,
                                 device=cuda_device)
    plan.set_chip_markers(case.x, case.y, case.fg_radius, case.chamber_radius, case.max_button_radius)
    ref = plan.run_device(case.tiles)
    image_ref, roi_ref, stats_ref = ref.image.cpu().contiguous(), ref.roi.cpu(), ref.stats.cpu()
    assert ref.image.is_contiguous() == (cc == 4)
    runner = pipeline.HostStagedRunner(plan)
    tiles_host = case.tiles.cpu().pin_memory()
    image_h, roi_h, stats_h = runner.alloc_host_outputs()
    for _ in range(3):                 # back-to-back assays reuse the device buffers safely
        image_h.zero_(); roi_h.zero_(); stats_h.zero_()
        runner.run(tiles_host, image_h, roi_h, stats_h)
        runner.synchronize()
        assert torch.equal(image_h.view(torch.int16), image_ref.view(torch.int16))
        assert torch.equal(roi_h.view(torch.int16), roi_ref.view(torch.int16))
        assert torch.equal(stats_h, stats_ref)
    assert runner.h2d_bytes == tiles_host.numel() * 2


def test_bead_plan_time_series(cuda_device):
    """Beads over several timepoints: masks are computed once and broadcast (find.py:585-586)."""
    from magnify_b200 import pipeline

    rng = np.random.default_rng(9)
    c, t, h, w, length = 3, 4, 256, 320, 50
    tiles = rng.integers(0, 65535, (c, t, 1, 1, h, w), dtype=np.uint16, endpoint=True)
    beads = np.stack([rng.integers(0, h, 25), rng.integers(0, w, 25), rng.integers(1, 14, 25)], 1).astype(np.float64)
    plan = pipeline.QuantifyPlan(tiles.shape, 0, length, device=cuda_device)
    plan.set_bead_markers(beads)
    res = plan.run_device(torch.from_numpy(tiles).to(cuda_device))
    image = o_st.stitch(tiles, 0)
    labels, fg, bg = o_rois.bead_masks(beads, h, w, length)
    x = np.repeat(beads[:, 1:2], t, 1)
    y = np.repeat(beads[:, 0:1], t, 1)
    roi = o_rois.gather_rois(image, x, y, length)
    np.testing.assert_array_equal(res.image.cpu().numpy(), image)
    np.testing.assert_array_equal(res.roi.cpu().numpy(), roi)
    np.testing.assert_array_equal(res.fg[:, 0].cpu().numpy().astype(bool), fg)
    want = o_red.masked_stats(roi, np.repeat(fg[:, None], t, 1), np.repeat(bg[:, None], t, 1))
    np.testing.assert_allclose(res.stats.cpu().numpy(), want, rtol=1e-12, equal_nan=True)


def test_chunk_stager_from_pageable_blocks(cuda_device):
    """Chunk provider -> pinned ring -> HBM (the dask-chunk staging loop): blocks arrive from
    pageable memory in arbitrary order; results equal the device-resident run."""
    from magnify_b200 import pipeline, synth

    case = synth.chip_case(c=2, t=3, r=2, cc=4, h=256, w=256, overlap=22, rows=3, cols=3, row_dist=126.1,
                           col_dist=250.0, seed=4, device=cuda_device)
    plan = pipeline.QuantifyPlan(case.tiles.shape, case.overlap, case.roi_length, case.flat, case.dark,
                                 device=cuda_device)
    plan.set_chip_markers(case.x, case.y, case.fg_radius, case.chamber_radius, case.max_button_radius)
    ref = plan.run_device(case.tiles)
    image_ref, roi_ref, stats_ref = ref.image.cpu(), ref.roi.cpu(), ref.stats.cpu()
    tiles_np = case.tiles.cpu().numpy()                      # pageable
    blocks = list(pipeline.iter_blocks(tiles_np))
    rng = np.random.default_rng(0)
    rng.shuffle(blocks)
    runner = pipeline.HostStagedRunner(plan)
    stager = pipeline.ChunkStager(runner, depth=2, threads=3)
    image_h, roi_h, stats_h = runner.alloc_host_outputs()
    for _ in range(2):
        assert stager.feed(iter(blocks)) == 6
        runner.finish(image_h, roi_h, stats_h)
        runner.synchronize()
        assert torch.equal(image_h.view(torch.int16), image_ref.view(torch.int16))
        assert torch.equal(roi_h.view(torch.int16), roi_ref.view(torch.int16))
        assert torch.equal(stats_h, stats_ref)
    stager.close()
    with pytest.raises(ValueError):
        stager2 = pipeline.ChunkStager(runner, depth=1, threads=1)
        stager2.feed(iter([((0, 0), np.zeros((1, 1, 8, 8), np.uint16))]))


def test_tiff_tiles_staged_through_pinned_ring(cuda_device, tmp_path):
    """Reader -> staging (SURVEY.md section 8f N2): one TIFF file per (channel, time, row, col),
    pages read natively into the pinned ring slots, then the same flat-field + stitch + gather as
    the device-resident run; also the `flatfield_correct` / `stitch` components on the lazy stack."""
    import os

    from magnify_b200 import pipeline, reader, synth
    from magnify_b200.components import FlatfieldStitcher
    from tiffgen import write_tiff

    case = synth.chip_case(c=2, t=3, r=2, cc=4, h=256, w=256, overlap=22, rows=3, cols=3, row_dist=126.1,
                           col_dist=250.0, seed=9, device=cuda_device)
    tiles_np = case.tiles.cpu().numpy()
    c, t, r, cc, h, w = tiles_np.shape
    for idx in np.ndindex(c, t, r, cc):
        write_tiff(os.path.join(tmp_path, f"chip_ch{idx[0]}_2024010{idx[1] + 1}-000000_{idx[2]}_{idx[3]}.tif"),
                   [tiles_np[idx]], rows_per_strip=[None, 64, 100][idx[3] % 3], big=bool(idx[2] % 2))
    (xp,) = list(reader.Reader(threads=4)(os.path.join(tmp_path, "chip_(channel)_(time)_(row)_(col).tif")))
    tiles = xp["tile"].data
    assert tiles.shape == tiles_np.shape

    plan = pipeline.QuantifyPlan(case.tiles.shape, case.overlap, case.roi_length, case.flat, case.dark,
                                 device=cuda_device)
    plan.set_chip_markers(case.x, case.y, case.fg_radius, case.chamber_radius, case.max_button_radius)
    ref = plan.run_device(case.tiles)
    image_ref, roi_ref, stats_ref = ref.image.cpu(), ref.roi.cpu(), ref.stats.cpu()
    runner = pipeline.HostStagedRunner(plan)
    stager = pipeline.ChunkStager(runner, depth=2, threads=2)
    image_h, roi_h, stats_h = runner.alloc_host_outputs()
    assert stager.feed(tiles.blocks()) == c * t
    runner.finish(image_h, roi_h, stats_h)
    runner.synchronize()
    stager.close()
    assert torch.equal(image_h.view(torch.int16), image_ref.view(torch.int16))
    assert torch.equal(roi_h.view(torch.int16), roi_ref.view(torch.int16))
    assert torch.equal(stats_h, stats_ref)

    # flat / dark given as TIFF files (preprocess.py:75-81), float64 pages
    flat_np, dark_np = np.asarray(case.flat), np.asarray(case.dark)
    if flat_np.ndim == 2:
        flat_arg = write_tiff(os.path.join(tmp_path, "flat.tif"), [flat_np], byteorder=">")
        dark_arg = write_tiff(os.path.join(tmp_path, "dark.tif"), [dark_np], big=True)
    else:
        flat_arg, dark_arg = flat_np, dark_np
    out = FlatfieldStitcher(flat_arg, dark_arg, case.overlap, device=cuda_device)(xp)
    np.testing.assert_array_equal(out.image.values, image_ref.numpy())


def test_markers_located_on_device_image(cuda_device):
    """tiles in HBM -> flat-field + stitch -> buttons found on the device image -> gather + stats,
    without the image leaving the GPU; equals the component path (image through the host)."""
    from magnify_b200 import pipeline
    from magnify_b200.components import BeadFinder, ButtonFinder, summaries
    from magnify_b200.dataset import Assay
    from test_gpu_finders import draw_beads, draw_chip
    from test_gpu_end_to_end import split_into_tiles

    shape, overlap, t = (5, 4), 8, 3
    chip = draw_chip(shape, 20, row_dist=100, col_dist=100) + 50                         # (600, 500)
    frames = np.stack([chip + 3 * k for k in range(t)])
    tiles = np.stack([split_into_tiles(f, 2, 2, overlap) for f in frames])[None]          # (1, T, 2, 2, h, w)
    tiles_d = torch.from_numpy(np.ascontiguousarray(tiles)).to(cuda_device)
    tag = np.full(shape, "default", dtype="<U200")
    kw = dict(row_dist=100, col_dist=100, min_button_diameter=16, max_button_diameter=32, chamber_diameter=60,
              num_iter=20000, min_roundness=0.2, cluster_penalty=50, search_timestep=[0, 2], device=cuda_device, seed=4)
    plan = pipeline.QuantifyPlan(tiles_d.shape, overlap, ButtonFinder(**kw).roi_length, device=cuda_device)
    image = plan.stitched(tiles_d)
    plan.locate_chip_markers(image, ButtonFinder(**kw), tag)
    res = plan.run_device(tiles_d, image=image)
    np.testing.assert_array_equal(res.image.cpu().numpy()[0], frames)
    assay = Assay({"image": (("channel", "time", "im_y", "im_x"), frames[None])},
                  coords={"channel": (("channel",), np.array(["c0"])), "tag": (("mark_row", "mark_col"), tag),
                          "valid": (("mark_row", "mark_col", "time"), np.ones(shape + (t,), bool))})
    out = ButtonFinder(**kw)(assay)
    np.testing.assert_array_equal(plan.x.cpu().numpy(), out.x.values)
    np.testing.assert_array_equal(res.roi.cpu().numpy(), out.roi.values)
    fg = res.fg.cpu().numpy().astype(bool)[:, res.mask_t.cpu().numpy()]
    np.testing.assert_array_equal(fg, out.fg.values)
    assert (res.stats[:, 0, :, 4].cpu().numpy() > 900).all()                              # fg means on the buttons
    # beads: the plan equals BeadFinder with the same centres on the same image
    beads_img = draw_beads((600, 500), [[100, 100], [300, 250], [500, 400]]) + 20
    tiles_b = torch.from_numpy(np.ascontiguousarray(split_into_tiles(beads_img, 2, 2, overlap)[None, None])).to(cuda_device)
    finder = BeadFinder(16, 24, num_iter=5000, device=cuda_device)
    bplan = pipeline.QuantifyPlan(tiles_b.shape, overlap, finder.roi_length, device=cuda_device)
    bimage = bplan.stitched(tiles_b)
    bplan.locate_bead_markers(bimage, finder)
    bres = bplan.run_device(tiles_b, image=bimage)
    assert bres.roi.shape[0] == 3 and (bres.stats[:, 0, 0, 4].cpu().numpy() > 900).all()
    bassay = Assay({"image": (("channel", "time", "im_y", "im_x"), bimage.cpu().numpy())},
                   coords={"channel": (("channel",), np.array(["c0"]))})
    beads = finder.find_centers(bassay, bimage)
    bout = BeadFinder(16, 24, centers=beads, device=cuda_device)(bassay)
    np.testing.assert_array_equal(bplan.x.cpu().numpy(), bout.x.values)
    np.testing.assert_array_equal(bres.roi.cpu().numpy(), bout.roi.values)
    mask_t = bres.mask_t.cpu().numpy()
    np.testing.assert_array_equal(bres.fg.cpu().numpy().astype(bool)[:, mask_t], bout.fg.values)
    np.testing.assert_array_equal(bres.bg.cpu().numpy().astype(bool)[:, mask_t], bout.bg.values)
    np.testing.assert_array_equal(bres.stats.cpu().numpy(), summaries(bout, device=cuda_device).cpu().numpy())


@pytest.mark.parametrize("identity", [False, True])
def test_streaming_runner_two_passes(cuda_device, tmp_path, identity):
    """Stacks larger than HBM: two sweeps over the block source with `depth` timepoints resident;
    per-timepoint results equal the all-resident run (from NumPy blocks and from TIFF pages)."""
    import os

    from magnify_b200 import pipeline, reader, synth
    from tiffgen import write_tiff

    case = synth.chip_case(c=2, t=5, r=2, cc=2, h=256, w=256, overlap=22, rows=3, cols=2, row_dist=126.1,
                           col_dist=200.0, seed=13, device=cuda_device)
    flat, dark = (1.0, 0.0) if identity else (case.flat, case.dark)
    plan = pipeline.QuantifyPlan(case.tiles.shape, case.overlap, case.roi_length, flat, dark, device=cuda_device)
    radius = np.repeat(case.fg_radius, 2, axis=1)
    plan.set_chip_markers(case.x, case.y, radius, case.chamber_radius, case.max_button_radius, search_timesteps=[0, 3])
    ref = plan.run_device(case.tiles)
    image_ref, roi_ref, stats_ref = ref.image.cpu().numpy(), ref.roi.cpu().numpy(), ref.stats.cpu().numpy()
    tiles_np = case.tiles.cpu().numpy()
    c, t = tiles_np.shape[:2]

    def check(source, depth):
        seen = []

        def sink(ti, image, roi, stats):
            seen.append(ti)
            np.testing.assert_array_equal(image, image_ref[:, ti])
            np.testing.assert_array_equal(roi, roi_ref[:, :, ti])
            np.testing.assert_array_equal(stats, stats_ref[:, :, ti])

        runner = pipeline.StreamingRunner(plan, depth=depth)
        runner.run(source, sink)
        assert seen == list(range(t))
        passes = 1 if identity else 2
        assert runner.h2d_bytes == passes * tiles_np.nbytes

    check(lambda ci, ti, dst: np.copyto(dst, tiles_np[ci, ti]), depth=2)
    check(lambda ci, ti, dst: np.copyto(dst, tiles_np[ci, ti]), depth=3)
    if not identity:
        for idx in np.ndindex(*tiles_np.shape[:4]):
            write_tiff(os.path.join(tmp_path, f"s_ch{idx[0]}_2024010{idx[1] + 1}-000000_{idx[2]}_{idx[3]}.tif"), [tiles_np[idx]])
        (xp,) = list(reader.Reader(threads=4)(os.path.join(tmp_path, "s_(channel)_(time)_(row)_(col).tif")))
        lazy = xp["tile"].data
        check(lambda ci, ti, dst: lazy.read((ci, ti), dst), depth=2)
    with pytest.raises(ValueError):
        pipeline.StreamingRunner(plan, depth=1)
