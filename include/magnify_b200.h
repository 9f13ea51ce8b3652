/* magnify_b200 -- C ABI of the B200-native per-marker quantification hot path.
 *
 * One shared library (magnify_b200/libmagnify_b200.so, built by __graft_entry__.build() with
 * nvcc -gencode arch=compute_100a,code=sm_100a).  Every entry point takes plain pointers and
 * sizes; pointers are DEVICE pointers unless the parameter name starts with `host_`.  All
 * launches go to the caller's stream (`stream` is a cudaStream_t passed as void*; NULL = the
 * legacy default stream) and return without synchronising.  Return value: 0 on success,
 * a negative MGB_E* code for argument errors (nothing launched), or a positive cudaError_t.
 *
 * The reference (FordyceLab/magnify v0.12.5) is pure Python; there is no FFI in it to mirror.
 * Each function below names the reference lines whose arithmetic it replaces; the Python
 * binding a magnify maintainer would add is in INTEGRATION.md (ctypes) and implemented in
 * magnify_b200/_lib.py.
 *
 * Array layouts (row-major, contiguous):
 *   tiles  (C, T, R, Cc, H, W)   the reference's canonical tile stack (preprocess.py:24)
 *   image  (C, T, Him, Wim)      stitched images, Him = R*(H-ov), Wim = Cc*(W-ov) (stitch.py:23-39);
 *                                rows may be padded: `image_pitch` = elements between row starts
 *                                (0 or Wim = dense).  A pitch that makes rows 16-byte aligned keeps
 *                                the vectorised kernels usable for any tile grid (e.g. 10x10 tiles
 *                                with overlap 102: Wim = 19460 is not a multiple of 8).
 *   boxes  (M, T, 2) int32       (top, left) of every marker's ROI at every timepoint
 *   roi    (M, C, T, L, L)       find.py:533 / find.py:89-92 after the stack at :182
 *   fg,bg  (M, Tm, L, L) uint8   0/1 masks; Tm = number of distinct mask timesteps
 *   stats  (M, C, T, 8) float64  n_fg, n_bg, sum_fg, sum_bg, mean_fg, mean_bg, median_fg, median_bg
 */
#ifndef MAGNIFY_B200_H
#define MAGNIFY_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MGB_ABI_VERSION 12

#define MGB_OK 0
#define MGB_EINVAL (-1)      /* bad argument (null pointer, negative size, bad itemsize ...) */
#define MGB_EALIGN (-2)      /* pointer / pitch does not meet the alignment a fast path needs */
#define MGB_EUNSUPPORTED (-3) /* shape or dtype outside what this build implements */
#define MGB_EIO (-4)         /* a file could not be opened or read (tiff staging) */
#define MGB_EFORMAT (-5)     /* not a TIFF / BigTIFF file, or its directory is inconsistent */

/* dtype codes for the generic (any-dtype) entry points */
#define MGB_U8 0
#define MGB_U16 1
#define MGB_F32 2
#define MGB_F64 3

int mgb_abi_version(void);
/* Human-readable text for a return code of this library (cudaGetErrorString for codes > 0). */
const char* mgb_error_string(int code);
/* Number of SMs of the current device (grid sizing / reporting). */
int mgb_sm_count(void);
/* Kernels launched by this library in this process so far (bench.py's gpu_launches). */
int64_t mgb_launch_count(void);

/* Experiment knob (tools/l2_reuse_probe.py): make [base, base+bytes) a persisting-L2 access-policy window of
 * `stream` (hit_ratio of its lines are kept, the rest stream through); base == NULL resets the stream's window
 * and hands the persisting lines back.  Results never depend on it. */
int mgb_l2_persist(void* stream, const void* base, int64_t bytes, float hit_ratio);

/* Tuning knob of the vectorised stitch / flat-field+stitch kernel: prefetch-ring depth x CTAs per
 * SM (0: 6x2 default, 1: 11x2, 2: 8x3).  Returns the previous value.  Results do not depend on it. */
int mgb_set_stitch_variant(int variant);

/* ---- F2: tile stitching, reference src/magnify/stitch.py:22-39 ----------------------------
 * image[c,t,y,x] = tiles[c,t, y/h, x/w, clip + y%h, clip + x%w], clip = overlap/2,
 * h = H-overlap, w = W-overlap.  Pure copy for any itemsize in {1,2,4,8}.  Argument checks
 * mirror stitch.py:8-9,16-20 (overlap < 0 or >= tile size -> MGB_EINVAL).  Picks a 128-bit
 * vectorised kernel when W*itemsize and image_pitch*itemsize are multiples of 16 bytes, else an
 * element-wise kernel; `used_fast` (host pointer, may be NULL) reports which. */
int mgb_stitch(const void* tiles, void* image, int64_t image_pitch, int64_t C, int64_t T, int64_t R,
               int64_t Cc, int64_t H, int64_t W, int64_t overlap, int itemsize, int* host_used_fast,
               void* stream);

/* ---- F1: flat-field correction, reference src/magnify/preprocess.py:83-87 -----------------
 * out = trunc((((max(float64(x) - dark, 0)) / flat) * M) / M2) with the two GLOBAL maxima
 * M = max(max(x - dark, 0)), M2 = max(max(x - dark, 0) / flat) over every tile pixel.
 * flat / dark are float64 tables (K, H, W), K = 1 (shared) or K = C (per channel); scalars
 * are expanded by the caller.  flat must be finite and > 0.
 *
 * Pass 1a: per-position maximum of the raw uint16 pixels over all tiles that share a table.
 * Exact because x -> max(x-d,0) and t -> t/f (f > 0) are monotone, so both maxima are attained
 * at the per-position maximum.  tiles is viewed as (C, P, HW) with P = T*R*Cc planes per
 * channel; `splits` CTAs share each position and write xmax_partial (splits, K, HW). */
int mgb_flatfield_tilemax_u16(const uint16_t* tiles, int64_t C, int64_t P, int64_t HW, int K,
                              int splits, uint16_t* xmax_partial, void* stream);
/* Pass 1b: maxima[0] = max(maxima[0], M), maxima[1] = max(maxima[1], M2) (device float64[2])
 * from the partial per-position maxima, in exact IEEE float64 (__dsub_rn / __ddiv_rn).  The
 * caller zero-initialises maxima (all values are >= 0); several calls (time chunks, channels)
 * accumulate into it with atomic max. */
int mgb_flatfield_maxima(const uint16_t* xmax_partial, int splits, int K, int64_t HW,
                         const double* flat, const double* dark, double* maxima, void* stream);
/* Any-dtype pass 1 (slow, exact): maxima over n elements of a (C, P, HW) stack. maxima must be
 * zero-initialised by the caller (values are >= 0); results are combined with atomic max so
 * several calls may accumulate into the same maxima. */
int mgb_flatfield_maxima_generic(const void* tiles, int dtype, int64_t C, int64_t P, int64_t HW,
                                 int K, const double* flat, const double* dark, double* maxima,
                                 void* stream);
/* Pass 2 preparation: per-position fast-path coefficients gain[k,p], bias[k,p] (float64) from
 * flat, dark and the (all-reduced) maxima.  The apply kernel evaluates one FMA per pixel,
 * s = (2^20 + x) * gain + bias, whose mantissa holds floor(v) in its high word and frac(v) in
 * its low word; pixels within 2^-24 of an integer (or with unusable coefficients, encoded here
 * as gain = 0, bias = 2^20 so that the guard always fires) are recomputed with the reference's
 * exact operation order. */
int mgb_flatfield_tables(const double* flat, const double* dark, int K, int64_t HW,
                         const double* maxima, double* gain, double* bias, void* stream);
/* Pass 2: flat-field apply fused with the stitch (read 2 B, write 2*phi B per tile pixel).
 * With overlap = 0 and R = Cc = 1 this is flat-field alone.  uint16 only; needs W % 8 == 0,
 * image_pitch % 8 == 0 and 16-byte aligned base pointers, else MGB_EALIGN (the caller
 * then uses mgb_flatfield_apply_generic + mgb_stitch). */
int mgb_flatfield_stitch_u16(const uint16_t* tiles, uint16_t* image, int64_t image_pitch, int64_t C,
                             int64_t T, int64_t R, int64_t Cc, int64_t H, int64_t W, int64_t overlap, int K,
                             const double* flat, const double* dark, const double* gain,
                             const double* bias, const double* maxima, void* stream);
/* Any-dtype exact flat-field apply in tile layout (no stitch): out[i] = cast(v(x[i])). */
int mgb_flatfield_apply_generic(const void* tiles, void* out, int dtype, int64_t C, int64_t P,
                                int64_t HW, int K, const double* flat, const double* dark,
                                const double* maxima, void* stream);

/* Pitched device <-> host copy (cudaMemcpy2DAsync): rows of `width_bytes` between buffers with
 * different row pitches, e.g. a padded device image into a dense pinned host array.  kind: 1 = host
 * to device, 2 = device to host, 3 = device to device. */
int mgb_copy2d_async(void* dst, int64_t dst_pitch_bytes, const void* src, int64_t src_pitch_bytes,
                     int64_t width_bytes, int64_t rows, int kind, void* stream);

/* ---- F3: bounding boxes, reference src/magnify/utils.py:55-80 and the callers' round() -----
 * boxes[i] = (top, left) of bounding_box(round(x[i]), round(y[i]), L, W, H) with Python's
 * round-half-even (find.py:163-164,328-329,371-372,574-575,595-596).  rel (nullable) receives
 * (round(y) - top, round(x) - left), the mask centre of find.py:380-381. */
int mgb_bounding_boxes(const double* x, const double* y, int64_t n, int L, int64_t W, int64_t H,
                       int32_t* boxes, int32_t* rel, void* stream);

/* The ROI gather has two implementations: windows staged through shared memory (TMA tensor copies
 * or cp.async chunks, re-aligned and stored with 128-bit stores) and plain load/store kernels used
 * when the image pitch is not a multiple of 16 bytes or the window does not fit shared memory.  This switch forces the
 * plain kernels (tests cover both); returns the previous setting.  Default: enabled. */
int mgb_set_tma_enabled(int enabled);
/* Loader of the staged gather: 0 = TMA tensor copy (cp.async.bulk.tensor, default), 1 = per-warp
 * cp.async 16-byte chunks.  Both measured within 1% of each other on B200 (DRAM fetches 128-byte
 * lines for the row fragments either way).  Adding 2 (values 2, 3) disables the warp-per-marker
 * kernel that otherwise handles many-marker / few-window shapes (bead screens).  Returns the
 * previous value; results do not depend on it. */
int mgb_set_gather_loader(int loader);

/* ---- F4 (+R): ROI gather, reference find.py:160-169, 324-334, 370-377, 589-602 -------------
 * roi[m,c,t] = image[c,t, top:top+L, left:left+L] for any itemsize in {1,2,4,8}.
 * order (M) int32, nullable: a permutation giving the order in which markers are processed (results
 * are independent of it).  Spatially sorted markers let windows that overlap or share DRAM lines
 * hit in L2 (dense bead screens). */
int mgb_roi_gather(const void* image, int64_t image_pitch, int64_t C, int64_t T, int64_t H, int64_t W,
                   int itemsize, const int32_t* boxes, const int32_t* order, int64_t M, int L, void* roi,
                   void* stream);
/* Gather fused with the masked reductions the consumers run (identify.py:76-80,
 * filter.py:21-22,51,74,82, README.md:21-22): uint16 only.  mask_t (T) int32 maps each timepoint to
 * its mask timestep in fg/bg (M, Tm, L, L) (beads: all 0, find.py:585-586; chip: the source
 * search timestep, find.py:151,172-173); any non-zero mask byte counts as set.  roi may be NULL
 * (summaries only).  stats (M,C,T,8) float64: counts, exact integer sums, mean = sum / count (NaN
 * for an empty mask, like nanmean), and the exact masked medians (mean of the two middle values
 * for even counts, NaN for an empty mask, like nanmedian).  stats must be 16-byte aligned.
 *
 * fg_count_max / bg_count_max: upper bounds of the number of set pixels in any fg / bg mask (from
 * mgb_mask_count_max, or -1 = unknown).  With bounds of at most 1024 / 2560 pixels the kernel
 * compacts each marker's masks into offset lists once and takes sums AND medians from the staged
 * window in the same pass (want_median != 0).  Otherwise (unknown or larger masks, unaligned
 * images, L > 256) the sums come from the dp2a / plain kernels and the two median columns are
 * left NaN: *host_median_done (host pointer, nullable) tells the caller which happened so that it
 * can run mgb_roi_median_u16 on the crops. */
int mgb_roi_gather_stats_u16(const uint16_t* image, int64_t image_pitch, int64_t C, int64_t T, int64_t H,
                             int64_t W, const int32_t* boxes, const int32_t* order, const int32_t* mask_t,
                             int64_t Tm, const uint8_t* fg, const uint8_t* bg, int64_t M, int L,
                             uint16_t* roi, double* stats, int want_median, int fg_count_max,
                             int bg_count_max, int* host_median_done, void* stream);
/* counts[0] = max over the n_masks fg masks of their non-zero bytes, counts[1] likewise for bg
 * (device int32[2]; mask_len = L*L bytes per mask). */
int mgb_mask_count_max(const uint8_t* fg, const uint8_t* bg, int64_t n_masks, int64_t mask_len,
                       int32_t* counts, void* stream);
/* Multi-GPU variant: the summaries are written by the kernel itself into the gathered buffer of
 * EVERY rank over NVLink peer memory (no separate all-gather).  host_peer_stats[j] (host array of
 * n_peers <= 8 device addresses) points at THIS rank's (M,C,T,8) block inside rank j's gathered
 * (ranks,M,C,T,8) buffer (peer-mapped, e.g. torch symmetric memory); the caller synchronises the
 * ranks afterwards.  Every peer address must be 16-byte aligned.  Needs the staged kernels (else
 * MGB_EUNSUPPORTED). */
int mgb_roi_gather_stats_peers_u16(const uint16_t* image, int64_t image_pitch, int64_t C, int64_t T,
                                   int64_t H, int64_t W, const int32_t* boxes, const int32_t* order, const int32_t* mask_t,
                                   int64_t Tm, const uint8_t* fg, const uint8_t* bg, int64_t M, int L,
                                   uint16_t* roi, const uint64_t* host_peer_stats, int n_peers,
                                   int want_median, int fg_count_max, int bg_count_max,
                                   int* host_median_done, void* stream);
/* The same summaries from an roi that already exists (the `quantify` component on a dataset
 * produced elsewhere): roi (M,C,T,L,L) uint16 -> stats (M,C,T,8), median columns NaN. */
int mgb_roi_stats_u16(const uint16_t* roi, int64_t M, int64_t C, int64_t T, int L,
                      const int32_t* mask_t, int64_t Tm, const uint8_t* fg, const uint8_t* bg,
                      double* stats, void* stream);
/* Exact masked median per (m,c,t) of a uint16 roi (M,C,T,L,L) (identify.py:79, filter.py:21-22):
 * mean of the two middle values for even counts, NaN for an empty mask, as np.nanmedian.  Any L
 * (keys in registers up to L = 160, re-read per bisection step above).  The result for ROI n goes
 * to median[n * median_stride] (1 = dense (M,C,T); 8 with median = stats + 6 / + 7 fills the
 * median columns of a stats buffer). */
int mgb_roi_median_u16(const uint16_t* roi, int64_t M, int64_t C, int64_t T, int L,
                       const int32_t* mask_t, int64_t Tm, const uint8_t* mask, double* median,
                       int64_t median_stride, void* stream);

/* The same two reductions for a float32 roi (the reference accepts float images, tests/test_chip.py:76-96):
 * float64 accumulation in a fixed order, NaN pixels skipped (nanmean / nanmedian); the median is the
 * exact middle value (mean of the two middle values for even counts) as float64. */
int mgb_roi_stats_f32(const float* roi, int64_t M, int64_t C, int64_t T, int L, const int32_t* mask_t, int64_t Tm,
                      const uint8_t* fg, const uint8_t* bg, double* stats, void* stream);
int mgb_roi_median_f32(const float* roi, int64_t M, int64_t C, int64_t T, int L, const int32_t* mask_t, int64_t Tm,
                       const uint8_t* mask, double* median, int64_t median_stride, void* stream);

/* ---- F8: chip masks, reference utils.py:30-52 through find.py:380-400 ----------------------
 * fg[m] = disc(radius r_fg[m]), bg[m] = annulus(r_inner < d <= r_outer) centred on rel[m] =
 * (y_rel, x_rel); cv.circle(thickness=-1) == {dx^2 + dy^2 <= r^2}.  counts (M,2) int32
 * (nullable) receives the fg/bg pixel counts. */
int mgb_chip_masks(const int32_t* rel, const int32_t* r_fg, int r_inner, int r_outer, int64_t M,
                   int L, uint8_t* fg, uint8_t* bg, int32_t* counts, void* stream);

/* ---- filter_nonround, reference filter.py:40-62 -------------------------------------------
 * perimeter[m] = sum over cv.findContours(mask m, RETR_EXTERNAL, CHAIN_APPROX_SIMPLE) of
 * cv.arcLength(contour, closed=True) for masks (M, L, L) uint8 (non-zero = foreground), L <= 160:
 * Suzuki-Abe border following, 8-connected, only outer borders whose parent is the frame; the
 * length is the sum of the chain steps (1 or sqrt 2) in float64 (OpenCV rounds each polygon
 * segment to float32: <= 6e-8 relative difference). */
int mgb_mask_perimeters(const uint8_t* masks, int64_t M, int L, double* perimeter, void* stream);

/* ---- F5-F7: bead masks, reference utils.py:380-465 and find.py:561-586 ---------------------
 * HOST helper: hw[0..r] = row half-widths of filled_circle_points(r) (utils.py:398-430). */
int mgb_disc_halfwidths(int r, int32_t* host_hw);
/* labels (H, W) int32: -1 none, i sole owner, -2 shared (utils.py:380-395).  beads (M,3) int32
 * rows (row, col, radius >= 1); hw (rmax+1, rmax+1) int32 table, row r = halfwidths of radius r. */
int mgb_bead_labels(const int32_t* beads, int64_t M, int64_t H, int64_t W, const int32_t* hw,
                    int rmax, int32_t* labels, void* stream);
/* fg[m] = (labels[box m] == m), bg[m] = (labels[box m] == -1)  (find.py:580-584); boxes (M,2). */
int mgb_bead_masks(const int32_t* labels, int64_t H, int64_t W, const int32_t* boxes, int64_t M,
                   int L, uint8_t* fg, uint8_t* bg, int32_t* counts, void* stream);

/* ---- N1 / N4: edge detection of the circle finder, reference utils.py:20-27, 113-139 --------
 * All of it integer / IEEE-exact, i.e. bit-identical to the NumPy + OpenCV calls of the reference.
 * Every entry point works on a BATCH of B independent images (B, H, W) (B <= 65535): one full
 * image for bead detection (find.py:476-491), thousands of 72 x 72 crops for the per-ROI button
 * refinement (find.py:339-360).
 *
 * to_uint8 (utils.py:20-27), per image: dst = uint8(255 * (x - min) / (max - min)) in float64,
 * truncated (all zero when max == min).  dtype is an MGB_* code; n = pixels per image; minmax
 * (B, 2) doubles on the device is scratch and holds (min, max) per image afterwards. */
int mgb_to_uint8(const void* src, int dtype, int64_t B, int64_t n, uint8_t* dst, double* minmax, void* stream);
/* cv.GaussianBlur(img, (5,5), 0) on uint8 followed by cv.Scharr(.., CV_32F, 1, 0) / (.., 0, 1)
 * (utils.py:114-118), BORDER_REFLECT_101.  The gradients are exact integers in [-4080, 4080] and
 * are stored as int16 (what utils.py:128-129 passes to Canny; float32 dx, dy are the same numbers). */
int mgb_edge_gradients_u8(const uint8_t* image, int64_t B, int64_t H, int64_t W, uint8_t* blurred, int16_t* dx,
                          int16_t* dy, void* stream);
/* Exact order statistics of m = dx^2 + dy^2 over the n pixels of every image:
 * host_values[b, i] = the host_ranks[i]-th smallest m (0-based) of image b, up to 4 ranks per
 * call.  grad = sqrt(float32(m)) (utils.py:119) is monotone in m, so these are the order
 * statistics np.quantile interpolates between (utils.py:125-126).  SYNCHRONISES the stream (three
 * histogram round trips).  scratch: B * 4 * (1 + 2048) uint32 on the device. */
int mgb_gradient_order_stats(const int16_t* dx, const int16_t* dy, int64_t B, int64_t n, const int64_t* host_ranks,
                             int n_ranks, int64_t* host_values, uint32_t* scratch, void* stream);
/* cv.Canny(dx, dy, threshold1, threshold2, L2gradient=True) (utils.py:127-133): edges (B,H,W)
 * uint8 0/1.  thresholds (B, 2) int32 on the device = the integer (low, high) OpenCV derives
 * (low = floor(min(t1,32767)^2), high likewise).  changed (1 int) is device scratch.  Non-maximum
 * suppression writes two bit planes (strong / candidate, one word per row and 32 pixels); the
 * hysteresis floods them one warp per 32x32 tile and is iterated to its fixed point,
 * SYNCHRONISING the stream once per sweep; host_sweeps (nullable) returns the sweep count. */
int mgb_canny(const int16_t* dx, const int16_t* dy, int64_t B, int64_t H, int64_t W, const int32_t* thresholds,
              uint8_t* edges, int* changed, int* host_sweeps, void* stream);

/* ---- N1 / N4: candidate circles and their scores, reference utils.py:141-189, 221-377 --------
 * Temporaries whose size is only known inside a call (CUB scan / sort storage, the unique-circle
 * list, the hysteresis activity maps) are taken from the device's default stream-ordered memory
 * pool (cudaMallocAsync); the library sets that pool's release threshold so that freed blocks are
 * kept for the next call instead of going back to the driver at every synchronisation.
 * Edge pixels grouped by grid cell (utils.py:347-377): counts / starts (B * cells + 1 int64 each,
 * cells = ceil(H/g) * ceil(W/g), cell-major per image) and coords (total uint32, row << 16 | col,
 * row-major inside a cell).  Call once with coords = NULL: counts and starts are computed and the
 * total is returned in *host_total (SYNCHRONISES the stream); then again, same arguments, with a
 * coords buffer of that capacity, which only fills the lists.  H, W <= 65535. */
int mgb_edge_cell_lists(const uint8_t* edges, int64_t B, int64_t H, int64_t W, int grid_length, int64_t* counts,
                        int64_t* starts, uint32_t* coords, int64_t coords_capacity, int64_t* host_total, void* stream);
/* num_iter circumcircles per image from three random edge pixels of one grid cell
 * (utils.py:288-344; arithmetic bit-identical to the reference's numba code, draws from a
 * counter-based generator keyed by `seed`, or from `randoms` (B, num_iter, 3) uint32 when given).
 * raw (B, num_iter, 3) float32 (nullable) receives (row, col, radius) of every draw.  When `table`
 * (table_capacity uint64, a power of two >= 2 * B * num_iter) is given, draws are filtered to
 * min_radius <= radius <= max_radius, rounded half-to-even, tested against the image
 * (utils.py:157-165) and de-duplicated: circles (<= B * num_iter, 4) int32 = (image, row, col,
 * radius), *host_n_unique of them, sorted by (image, row, col, radius).  counter: one uint64 of device scratch.
 * SYNCHRONISES the stream when `table` is given. */
int mgb_sample_circles(const uint32_t* coords, const int64_t* starts, const int64_t* counts, int64_t B, int64_t H,
                       int64_t W, int grid_length, int64_t num_iter, float min_radius, float max_radius,
                       uint64_t seed, const uint32_t* randoms, float* raw, uint64_t* table, int64_t table_capacity,
                       int32_t* circles, int64_t* host_n_unique, unsigned long long* counter, void* stream);
/* angle = float32(atan2(dy, dx)) per pixel (utils.py:169); with `edges` (nullable, n uint8) only
 * at edge pixels, 0 elsewhere -- the score never reads the angle of a non-edge pixel. */
int mgb_gradient_angles(const int16_t* dx, const int16_t* dy, const uint8_t* edges, int64_t n, float* angle,
                        void* stream);
/* HOST: perimeter of the reference's circle raster (utils.py:433-465) in the reference's order,
 * (drow, dcol) pairs; capacity >= 20 * r points. */
int mgb_circle_perimeter(int r, int four_connected, int32_t* host_points, int capacity, int* host_n);
/* scores[i] = mean_grad(...)[i] / len(perimeter) of utils.py:181-183, 221-249 for circles (N, 4)
 * int32 (image, row, col, radius) with rmin <= radius <= rmax (NaN otherwise).  perim_offsets
 * (rmax - rmin + 2), perim_points (P, 2) int16, perim_expected (P) float64 = arctan2(drow, dcol)
 * concatenate the perimeters of radius rmin..rmax. */
int mgb_score_circles(const int32_t* circles, int64_t N, int64_t H, int64_t W, const uint8_t* edges,
                      const float* angle, int rmin, int rmax, const int32_t* perim_offsets,
                      const int16_t* perim_points, const double* perim_expected, float* scores, void* stream);
/* order (N) int32: the permutation that lists circles (N, 4) image by image, best score first
 * (utils.py:192-193, `argsort(-scores)`), equal scores in input order (stable). */
int mgb_order_circles(const int32_t* circles, const float* scores, int64_t N, int32_t* order, void* stream);
/* utils.py:252-285 on the device for circles (N, 4) int32 (image, row, col, radius) listed image by
 * image, best first (the output order of mgb_order_circles), centres within max_radius of a
 * B x H x W batch: state[i] = 1 when circle i survives, 2 when it is suppressed.  Two circles
 * conflict when the rings of radius min_dist around their centres share a pixel, which depends
 * only on the centre offset: conflict is that relation as a (4 min_dist + 1)^2 byte map on the
 * device (index (drow + 2 min_dist) * (4 min_dist + 1) + dcol + 2 min_dist).  The sequential
 * best-first pass is reproduced by rounds of "rejected once a higher-ranked conflicting circle is
 * kept, kept once all of them are rejected"; SYNCHRONISES the stream once per round and returns
 * MGB_EUNSUPPORTED (state undefined) when 256 rounds did not settle every circle.  Callers must
 * use the host version when a centre lies more than min_dist + 1 pixels outside the image (there
 * the reference's raster indices wrap around). */
int mgb_filter_neighbors_device(const int32_t* circles, int64_t N, int64_t B, int64_t H, int64_t W, int max_radius,
                                int min_dist, const uint8_t* conflict, uint8_t* state, int* host_rounds, void* stream);
/* HOST: utils.py:252-285 on circles (n, 3) int32 (row, col, radius) sorted best first:
 * host_valid[i] = 1 when circle i survives. */
int mgb_filter_neighbors(const int32_t* host_circles, int64_t n, int min_dist, uint8_t* host_valid);

/* ---- S / N2: TIFF page staging, reference src/magnify/reader.py:265-279 ---------------------
 * HOST-ONLY entry points (no kernel is launched): the reference's lazy tile loader reads one
 * TIFF page per dask chunk with `tifffile.TiffFile(f).pages[i].asarray()`.  These read the same
 * page bytes -- classic TIFF and BigTIFF, either byte order, strips or tiles, Compression 1
 * (direct pread), 5 (LZW), 8 / 32946 (Deflate) or 32773 (PackBits), Predictor 1 or 2 -- straight
 * into caller-owned host memory (normally a pinned staging buffer that the next
 * cudaMemcpyAsync consumes), byte-swapped to host order.  A page is returned as `height` rows of
 * `width * samples` items in file order, i.e. the (tile_y, tile_x) array `asarray()` gives.
 *
 * mgb_tiff_open parses the whole main IFD chain once.  info (12 x int64): width, height,
 * bits per sample, samples per pixel, SampleFormat (1 uint, 2 int, 3 float), Compression,
 * page bytes, support status (MGB_OK or the MGB_E* code a read would return), ImageDescription
 * length in bytes, strip count, 1 if BigTIFF, 1 if big-endian. */
int mgb_tiff_open(const char* host_path, void** host_handle);
int mgb_tiff_close(void* host_handle);
int mgb_tiff_page_count(const void* host_handle, int64_t* host_count);
int mgb_tiff_page_info(const void* host_handle, int64_t page, int64_t* host_info);
/* Raw ImageDescription bytes (tag 270: OME-XML / Micro-Manager metadata, reader.py:216-222). */
int mgb_tiff_description(const void* host_handle, int64_t page, char* host_buf, int64_t capacity);
/* Pages host_pages[0..n) of one open file into host_dst + i*dst_stride_bytes, `threads` readers. */
int mgb_tiff_read_pages(const void* host_handle, const int64_t* host_pages, int64_t n_pages, void* host_dst,
                        int64_t dst_stride_bytes, int threads);
/* Page `page` of each of n_files files (one file per (channel,time,row,col) index, the layout
 * reader.py:173-186 assembles from the path pattern) into host_dst + i*dst_stride_bytes.  Every
 * page must be width x height, single-sample, `bits` wide, else MGB_EFORMAT. */
int mgb_tiff_read_files(const char* const* host_paths, int64_t n_files, int64_t page, int64_t width, int64_t height,
                        int bits, void* host_dst, int64_t dst_stride_bytes, int threads);

/* Results to disk (no counterpart in the reference, which caches to zarr, accessor.py:18-35): n_pages
 * host pages of height x width items (bits in {8,16,32,64}; sample_format 1 uint, 2 int, 3 float) as
 * an uncompressed little-endian TIFF, one strip per page, written with `threads` parallel pwrite
 * calls.  bigtiff: 1 BigTIFF, 0 classic (MGB_EINVAL beyond 4 GB), -1 choose by size.
 * host_description (nullable) becomes the ImageDescription of the first page. */
int mgb_tiff_write(const char* host_path, const void* host_pages, int64_t n_pages, int64_t height, int64_t width,
                   int bits, int sample_format, int bigtiff, const char* host_description, int threads);

#ifdef __cplusplus
}
#endif
#endif /* MAGNIFY_B200_H */
