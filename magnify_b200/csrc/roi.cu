// F3 / F4 / R: bounding boxes, ROI gather and masked per-ROI reductions, hand-written for
// sm_100a.  Reference: src/magnify/utils.py:55-80 (bounding_box), find.py:160-169, 324-334,
// 370-377, 589-602 (crop loops), identify.py:76-80 and filter.py:21-22,51 (reductions).
//
// HBM layout: image (C,T,H,W), roi (M,C,T,L,L), masks (M,Tm,L,L) uint8, stats (M,C,T,6) f64.
// One CTA copies one ROI (m,c,t); CTAs are numbered in roi memory order so consecutive CTAs
// write consecutive 2*L*L-byte blocks.  Reductions ride on the copy: the pixels are already in
// registers, the masks (shared by all channels / copy-forward timepoints) come from L2.
#include "common.cuh"

namespace mgb {

// ---- F3 ------------------------------------------------------------------------------------
__device__ __forceinline__ void box_1d(long long c, int L, long long size, long long* lo) {
  long long a = c - L / 2;
  long long b = c + (L + 1) / 2;   // ceildiv(L, 2), utils.py:55-57
  if (a < 0) { b -= a; a = 0; }
  if (b > size) { a -= b - size; }
  *lo = a;
}

__global__ void __launch_bounds__(kThreads)
bounding_boxes_kernel(const double* __restrict__ x, const double* __restrict__ y, int64_t n, int L,
                      int64_t W, int64_t H, int32_t* __restrict__ boxes, int32_t* __restrict__ rel) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  // Python round() on a float64 is round-half-to-even == cvt.rni.
  const long long xr = __double2ll_rn(x[i]);
  const long long yr = __double2ll_rn(y[i]);
  long long top, left;
  box_1d(yr, L, H, &top);
  box_1d(xr, L, W, &left);
  boxes[2 * i] = (int32_t)top;
  boxes[2 * i + 1] = (int32_t)left;
  if (rel) {
    rel[2 * i] = (int32_t)(yr - top);
    rel[2 * i + 1] = (int32_t)(xr - left);
  }
}

// ---- F4 (+R) -------------------------------------------------------------------------------
struct GatherParams {
  const uint16_t* image;   // 16-bit units
  uint16_t* roi;           // may be null when STATS
  int64_t C, T, H, W;      // W = image row pitch in 16-bit units (>= logical width)
  const int32_t* boxes;    // (M,T,2) in elements; null = every box at (0, 0)
  int64_t marker_stride;   // 16-bit units between markers' images (0: all markers share `image`)
  int unit;                // 16-bit units per element (itemsize / 2)
  int L;                   // roi side in elements
  int Lu;                  // roi row length in 16-bit units
  uint32_t half;           // Lu / 2 words per row
  uint32_t magic;          // ceil(2^32 / half)
  uint32_t words;          // L * half
  const int32_t* mask_t;
  int64_t Tm;
  const uint8_t* fg;
  const uint8_t* bg;
  double* stats;
};

constexpr int kRec = 8;   // doubles per summary record: n_fg n_bg sum_fg sum_bg mean_fg mean_bg median_fg median_bg

__device__ __forceinline__ uint64_t block_sum_u64(uint64_t v, uint64_t* smem) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) smem[w] = v;
  __syncthreads();
  uint64_t s = 0;
#pragma unroll
  for (int i = 0; i < kThreads / 32; ++i) s += smem[i];
  return s;
}

// The median columns are left NaN: the caller fills them (roi_median kernels) when it wants them.
__device__ __forceinline__ void write_record(double* o, uint64_t na, uint64_t nb, uint64_t a, uint64_t b) {
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  o[0] = (double)na;
  o[1] = (double)nb;
  o[2] = (double)a;
  o[3] = (double)b;
  o[4] = (double)a / (double)na;   // 0/0 -> NaN, like nanmean over an empty mask
  o[5] = (double)b / (double)nb;
  o[6] = nan;
  o[7] = nan;
}

// Word path: 2 x 16-bit units per thread step (Lu even).  ALIGNED: source words 4-byte aligned.
template <bool STATS>
__global__ void __launch_bounds__(kThreads) roi_gather_words_kernel(const GatherParams p) {
  __shared__ uint64_t red[4][kThreads / 32];
  const int64_t n = blockIdx.x;                 // (m*C + c)*T + t
  const int64_t t = n % p.T;
  const int64_t c = (n / p.T) % p.C;
  const int64_t m = n / (p.T * p.C);
  const int32_t top = p.boxes ? p.boxes[(m * p.T + t) * 2] : 0;
  const int32_t left = p.boxes ? p.boxes[(m * p.T + t) * 2 + 1] : 0;
  const uint16_t* src = p.image + m * p.marker_stride + ((c * p.T + t) * p.H + top) * p.W + (int64_t)left * p.unit;
  const bool aligned = ((reinterpret_cast<uintptr_t>(src) & 3u) == 0) && ((p.W & 1) == 0);
  uint32_t* dst = p.roi ? reinterpret_cast<uint32_t*>(p.roi + n * (int64_t)p.L * p.Lu) : nullptr;
  const uint16_t* fgp = nullptr;
  const uint16_t* bgp = nullptr;
  if constexpr (STATS) {
    const int64_t mo = (m * p.Tm + p.mask_t[t]) * (int64_t)p.L * p.L;
    fgp = reinterpret_cast<const uint16_t*>(p.fg + mo);
    bgp = reinterpret_cast<const uint16_t*>(p.bg + mo);
  }
  // per-thread sums in 64 bits: a thread sees up to L*L/256 pixel pairs of up to 2 * 65535 each
  uint64_t s_fg = 0, s_bg = 0;
  uint32_t n_fg = 0, n_bg = 0;
  for (uint32_t w = threadIdx.x; w < p.words; w += kThreads) {
    const uint32_t row = __umulhi(w, p.magic);
    const uint32_t col = w - row * p.half;
    const uint16_t* sp = src + (int64_t)row * p.W + 2 * col;
    uint32_t v;
    if (aligned) {
      v = __ldg(reinterpret_cast<const uint32_t*>(sp));
    } else {
      v = (uint32_t)__ldg(sp) | ((uint32_t)__ldg(sp + 1) << 16);
    }
    if (dst) dst[w] = v;
    if constexpr (STATS) {
      // two mask bytes; any non-zero byte counts as set
      const uint32_t mf = __vcmpne4((uint32_t)__ldg(fgp + w), 0u) & 0x0101u;
      const uint32_t mb = __vcmpne4((uint32_t)__ldg(bgp + w), 0u) & 0x0101u;
      s_fg += __dp2a_lo(v, mf, 0u);
      s_bg += __dp2a_lo(v, mb, 0u);
      n_fg += __popc(mf);
      n_bg += __popc(mb);
    }
  }
  if constexpr (STATS) {
    const uint64_t a = block_sum_u64(s_fg, red[0]);
    const uint64_t b = block_sum_u64(s_bg, red[1]);
    const uint64_t na = block_sum_u64(n_fg, red[2]);
    const uint64_t nb = block_sum_u64(n_bg, red[3]);
    if (threadIdx.x == 0) write_record(p.stats + n * kRec, na, nb, a, b);
  }
}

// Scalar path: any unit type, any L (odd L, itemsize 1).
template <typename U, bool STATS>
__global__ void __launch_bounds__(kThreads)
roi_gather_scalar_kernel(const U* __restrict__ image, U* __restrict__ roi, int64_t C, int64_t T,
                         int64_t H, int64_t W, const int32_t* __restrict__ boxes, int64_t marker_stride, int L,
                         const int32_t* __restrict__ mask_t, int64_t Tm,
                         const uint8_t* __restrict__ fg, const uint8_t* __restrict__ bg,
                         double* __restrict__ stats) {
  __shared__ uint64_t red[4][kThreads / 32];
  const int64_t n = blockIdx.x;
  const int64_t t = n % T;
  const int64_t c = (n / T) % C;
  const int64_t m = n / (T * C);
  const int32_t top = boxes ? boxes[(m * T + t) * 2] : 0;
  const int32_t left = boxes ? boxes[(m * T + t) * 2 + 1] : 0;
  const U* src = image + m * marker_stride + ((c * T + t) * H + top) * W + left;
  U* dst = roi ? roi + n * (int64_t)L * L : nullptr;
  const uint8_t* fgp = nullptr;
  const uint8_t* bgp = nullptr;
  if constexpr (STATS) {
    const int64_t mo = (m * Tm + mask_t[t]) * (int64_t)L * L;
    fgp = fg + mo;
    bgp = bg + mo;
  }
  uint64_t s_fg = 0, s_bg = 0;
  uint32_t n_fg = 0, n_bg = 0;
  const int total = L * L;
  for (int i = threadIdx.x; i < total; i += kThreads) {
    const int row = i / L, col = i - row * L;
    const U v = src[(int64_t)row * W + col];
    if (dst) dst[i] = v;
    if constexpr (STATS) {
      const uint32_t f = fgp[i], b = bgp[i];
      s_fg += f ? (uint64_t)v : 0u;
      s_bg += b ? (uint64_t)v : 0u;
      n_fg += f ? 1u : 0u;
      n_bg += b ? 1u : 0u;
    }
  }
  if constexpr (STATS) {
    const uint64_t a = block_sum_u64(s_fg, red[0]);
    const uint64_t b = block_sum_u64(s_bg, red[1]);
    const uint64_t na = block_sum_u64(n_fg, red[2]);
    const uint64_t nb = block_sum_u64(n_bg, red[3]);
    if (threadIdx.x == 0) write_record(stats + n * kRec, na, nb, a, b);
  }
}

// ---- masked median (exact) -----------------------------------------------------------------
// Pixel <-> 32-bit search key (monotone; 0xffffffff = "not in the mask").  float32: the usual
// sign-flip order on the bit pattern; NaN pixels are skipped like np.nanmedian skips them.
__device__ __forceinline__ uint32_t median_key(uint16_t v) { return v; }
__device__ __forceinline__ uint32_t median_key(float v) {
  if (v != v) return 0xffffffffu;
  const uint32_t u = __float_as_uint(v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
template <typename TPix> __device__ __forceinline__ double median_value(uint32_t key);
template <> __device__ __forceinline__ double median_value<uint16_t>(uint32_t key) { return (double)key; }
template <> __device__ __forceinline__ double median_value<float>(uint32_t key) {
  return (double)__uint_as_float((key & 0x80000000u) ? (key & 0x7fffffffu) : ~key);
}

// One CTA per ROI.  Every thread keeps its pixels as 32-bit keys (masked-out -> 0xffffffff) in
// registers; the k-th smallest is found by a binary search on the key with one block count per
// step.  NPT = keys per thread.
template <int NPT, typename TPix>
__global__ void __launch_bounds__(kThreads)
roi_median_kernel(const TPix* __restrict__ roi, int64_t C, int64_t T, int L,
                      const int32_t* __restrict__ mask_t, int64_t Tm,
                      const uint8_t* __restrict__ mask, double* __restrict__ median, int64_t stride) {
  __shared__ uint32_t red[2][kThreads / 32];
  const int64_t n = blockIdx.x;
  const int64_t t = n % T;
  const int64_t m = n / (T * C);
  const int total = L * L;
  const TPix* src = roi + n * (int64_t)total;
  const uint8_t* mk = mask + (m * Tm + mask_t[t]) * (int64_t)total;
  uint32_t key[NPT];
  uint32_t cnt = 0;
#pragma unroll
  for (int i = 0; i < NPT; ++i) {
    const int idx = threadIdx.x + i * kThreads;
    key[i] = 0xffffffffu;
    if (idx < total && mk[idx]) {
      key[i] = median_key(src[idx]);
      if (key[i] != 0xffffffffu) ++cnt;
    }
  }
  int buf = 0;
  auto block_count = [&](uint32_t c) -> uint32_t {
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0) red[buf][threadIdx.x >> 5] = c;
    __syncthreads();
    uint32_t s = 0;
#pragma unroll
    for (int i = 0; i < kThreads / 32; ++i) s += red[buf][i];
    buf ^= 1;
    return s;
  };
  const uint32_t nvalid = block_count(cnt);
  if (nvalid == 0) {
    if (threadIdx.x == 0) median[n * stride] = __longlong_as_double(0x7ff8000000000000LL);
    return;
  }
  const uint32_t k1 = (nvalid - 1) >> 1;  // lower middle (0-based)
  // narrow the search to [min, max] of the masked values: real backgrounds span a few dozen grey
  // levels, so this replaces most of the 16 bisection steps by two block reductions
  uint32_t lo, hi;
  {
    uint32_t mn = 0xffffffffu, mx = 0;
#pragma unroll
    for (int i = 0; i < NPT; ++i) {
      mn = min(mn, key[i]);
      if (key[i] != 0xffffffffu) mx = max(mx, key[i]);
    }
    mn = __reduce_min_sync(0xffffffffu, mn);
    mx = __reduce_max_sync(0xffffffffu, mx);
    __shared__ uint32_t rng[2][kThreads / 32];
    if ((threadIdx.x & 31) == 0) { rng[0][threadIdx.x >> 5] = mn; rng[1][threadIdx.x >> 5] = mx; }
    __syncthreads();
    lo = 0xffffffffu; hi = 0;
#pragma unroll
    for (int i = 0; i < kThreads / 32; ++i) { lo = min(lo, rng[0][i]); hi = max(hi, rng[1][i]); }
  }
  while (lo < hi) {
    const uint32_t mid = lo + ((hi - lo) >> 1);   // float keys use the full 32 bits: lo + hi would wrap
    uint32_t c = 0;
#pragma unroll
    for (int i = 0; i < NPT; ++i) c += (key[i] <= mid) ? 1u : 0u;
    const uint32_t tot = block_count(c);
    if (tot >= k1 + 1) hi = mid; else lo = mid + 1;
  }
  const uint32_t v1 = lo;
  uint32_t v2 = v1;
  if ((nvalid & 1u) == 0) {
    // upper middle: v1 again if enough copies, else the smallest value above v1
    uint32_t c = 0, mn = 0xffffffffu;
#pragma unroll
    for (int i = 0; i < NPT; ++i) {
      c += (key[i] <= v1) ? 1u : 0u;
      if (key[i] > v1) mn = min(mn, key[i]);
    }
    const uint32_t tot = block_count(c);
    mn = __reduce_min_sync(0xffffffffu, mn);
    if ((threadIdx.x & 31) == 0) red[buf][threadIdx.x >> 5] = mn;
    __syncthreads();
    uint32_t g = 0xffffffffu;
#pragma unroll
    for (int i = 0; i < kThreads / 32; ++i) g = min(g, red[buf][i]);
    if (tot < k1 + 2) v2 = g;
  }
  if (threadIdx.x == 0) median[n * stride] = 0.5 * (median_value<TPix>(v1) + median_value<TPix>(v2));
}

// Any L: the keys do not fit in registers, so every bisection step re-reads the window (it stays
// in L2: at most 16 + 3 passes for uint16, 32 + 3 for float32).  One CTA per ROI.
template <typename TPix>
__global__ void __launch_bounds__(kThreads)
roi_median_big_kernel(const TPix* __restrict__ roi, int64_t C, int64_t T, int L, const int32_t* __restrict__ mask_t,
                      int64_t Tm, const uint8_t* __restrict__ mask, double* __restrict__ median, int64_t stride) {
  __shared__ uint32_t red[3][kThreads / 32];
  const int64_t n = blockIdx.x;
  const int64_t t = n % T;
  const int64_t m = n / (T * C);
  const int total = L * L;
  const TPix* src = roi + n * (int64_t)total;
  const uint8_t* mk = mask + (m * Tm + mask_t[t]) * (int64_t)total;
  // one block-wide pass: count of keys <= bound, smallest key > bound, and (first == true) min / max
  auto sweep = [&](uint32_t bound, uint32_t* count, uint32_t* above, uint32_t* lowest) {
    uint32_t c = 0, a = 0xffffffffu, lo = 0xffffffffu;
    for (int i = threadIdx.x; i < total; i += kThreads) {
      if (!mk[i]) continue;
      const uint32_t k = median_key(src[i]);
      if (k == 0xffffffffu) continue;
      c += (k <= bound) ? 1u : 0u;
      if (k > bound) a = min(a, k);
      lo = min(lo, k);
    }
    c = __reduce_add_sync(0xffffffffu, c);
    a = __reduce_min_sync(0xffffffffu, a);
    lo = __reduce_min_sync(0xffffffffu, lo);
    __syncthreads();   // the previous sweep's readers are done with `red`
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = c; red[1][threadIdx.x >> 5] = a; red[2][threadIdx.x >> 5] = lo; }
    __syncthreads();
    uint32_t sc = 0, sa = 0xffffffffu, sl = 0xffffffffu;
#pragma unroll
    for (int i = 0; i < kThreads / 32; ++i) { sc += red[0][i]; sa = min(sa, red[1][i]); sl = min(sl, red[2][i]); }
    *count = sc; *above = sa; *lowest = sl;
  };
  uint32_t nvalid, above, lo;
  sweep(0xfffffffeu, &nvalid, &above, &lo);     // every valid key is <= 0xfffffffe
  if (nvalid == 0) {
    if (threadIdx.x == 0) median[n * stride] = __longlong_as_double(0x7ff8000000000000LL);
    return;
  }
  const uint32_t k1 = (nvalid - 1) >> 1;
  uint32_t hi = 0xfffffffeu, cnt, dummy;
  if (sizeof(TPix) == 2) hi = 0xffffu;
  while (lo < hi) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    sweep(mid, &cnt, &above, &dummy);
    if (cnt >= k1 + 1) hi = mid; else lo = mid + 1;
  }
  uint32_t v2 = lo;
  if ((nvalid & 1u) == 0) {
    sweep(lo, &cnt, &above, &dummy);
    if (cnt < k1 + 2) v2 = above;
  }
  if (threadIdx.x == 0) median[n * stride] = 0.5 * (median_value<TPix>(lo) + median_value<TPix>(v2));
}

// Masked sums of a float32 roi: one CTA per (m, c, t), float64 accumulation in a fixed order
// (thread-strided partial sums, warp shuffles, then the warps in index order), NaN pixels skipped
// like np.nansum / np.nanmean.  Record layout as for uint16: n_fg, n_bg, sum_fg, sum_bg, mean_fg, mean_bg.
__global__ void __launch_bounds__(kThreads)
roi_stats_f32_kernel(const float* __restrict__ roi, int64_t C, int64_t T, int L, const int32_t* __restrict__ mask_t,
                     int64_t Tm, const uint8_t* __restrict__ fg, const uint8_t* __restrict__ bg,
                     double* __restrict__ stats) {
  __shared__ double red[4][kThreads / 32];
  const int64_t n = blockIdx.x;
  const int64_t t = n % T;
  const int64_t m = n / (T * C);
  const int total = L * L;
  const float* src = roi + n * (int64_t)total;
  const int64_t moff = (m * Tm + mask_t[t]) * (int64_t)total;
  double v[4] = {0.0, 0.0, 0.0, 0.0};   // n_fg, n_bg, sum_fg, sum_bg
  for (int i = threadIdx.x; i < total; i += kThreads) {
    const float x = src[i];
    if (x != x) continue;
    if (fg[moff + i]) { v[0] += 1.0; v[2] += (double)x; }
    if (bg[moff + i]) { v[1] += 1.0; v[3] += (double)x; }
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_down_sync(0xffffffffu, v[k], o);
    if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = v[k];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    for (int w = 0; w < kThreads / 32; ++w)
      for (int k = 0; k < 4; ++k) s[k] += red[k][w];
    double* out = stats + n * kRec;
    out[0] = s[0]; out[1] = s[1]; out[2] = s[2]; out[3] = s[3];
    out[4] = s[2] / s[0];   // 0 / 0 = NaN for an empty mask, like np.nanmean
    out[5] = s[3] / s[1];
    out[6] = out[7] = __longlong_as_double(0x7ff8000000000000LL);   // medians: filled by the median kernel
  }
}

static uint32_t magic_for(uint32_t d) { return (uint32_t)((0x100000000ULL + d - 1) / d); }

// roi_tma.cu
int roi_gather_tma(const void* image, int64_t pitch, int64_t C, int64_t T, int64_t H, int64_t W, int itemsize,
                   const int32_t* boxes, const int32_t* order, const int32_t* mask_t, int64_t Tm, const uint8_t* fg,
                   const uint8_t* bg, int64_t M, int L, void* roi, double* stats, const uint64_t* host_peers,
                   int n_peers, cudaStream_t st);

// roi_lists.cu
int roi_gather_lists(const void* image, int64_t pitch, int64_t C, int64_t T, int64_t H, int64_t W,
                     const int32_t* boxes, const int32_t* order, const int32_t* mask_t, int64_t Tm, const uint8_t* fg,
                     const uint8_t* bg, int64_t M, int L, void* roi, double* stats, int want_median, int nf_max,
                     int nb_max, const uint64_t* host_peers, int n_peers, cudaStream_t st);

extern int g_gather_loader;
extern int g_gather_wpm;

static int g_tma_enabled = 1;

}  // namespace mgb

using namespace mgb;

template <typename TPix>
static int launch_roi_median(const TPix* roi, int64_t M, int64_t C, int64_t T, int L, const int32_t* mask_t, int64_t Tm,
                             const uint8_t* mask, double* median, int64_t stride, void* stream) {
  if (M < 0 || C < 0 || T < 0 || L <= 0 || stride < 1) return MGB_EINVAL;
  const int64_t n_roi = M * C * T;
  if (n_roi == 0) return MGB_OK;
  if (n_roi > INT32_MAX) return MGB_EUNSUPPORTED;
  if (!roi || !mask_t || !mask || !median || Tm <= 0) return MGB_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  const int npt = (int)ceil_div((int64_t)L * L, kThreads);
#define MGB_MED(N) roi_median_kernel<N, TPix><<<(unsigned)n_roi, kThreads, 0, st>>>(roi, C, T, L, mask_t, Tm, mask, median, stride)
  if (npt <= 4) MGB_MED(4);
  else if (npt <= 10) MGB_MED(10);
  else if (npt <= 21) MGB_MED(21);
  else if (npt <= 40) MGB_MED(40);
  else if (npt <= 64) MGB_MED(64);
  else if (npt <= 100) MGB_MED(100);
  else roi_median_big_kernel<TPix><<<(unsigned)n_roi, kThreads, 0, st>>>(roi, C, T, L, mask_t, Tm, mask, median, stride);   // L > 160
#undef MGB_MED
  MGB_CUDA_LAUNCH_CHECK();
  return MGB_OK;
}

extern "C" {

int mgb_bounding_boxes(const double* x, const double* y, int64_t n, int L, int64_t W, int64_t H,
                       int32_t* boxes, int32_t* rel, void* stream) {
  if (n < 0 || L <= 0 || W < L || H < L || W > INT32_MAX || H > INT32_MAX) return MGB_EINVAL;
  if (n == 0) return MGB_OK;
  if (!x || !y || !boxes) return MGB_EINVAL;
  bounding_boxes_kernel<<<(unsigned)ceil_div(n, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
      x, y, n, L, W, H, boxes, rel);
  MGB_CUDA_LAUNCH_CHECK();
  return MGB_OK;
}

static int gather_common(const void* image, int64_t image_pitch, int64_t C, int64_t T, int64_t H, int64_t W,
                         int itemsize, const int32_t* boxes, const int32_t* order, int64_t marker_stride, const int32_t* mask_t, int64_t Tm, const uint8_t* fg,
                         const uint8_t* bg, int64_t M, int L, void* roi, double* stats,
                         cudaStream_t st, const uint64_t* host_peers = nullptr, int n_peers = 0,
                         int want_median = 0, int nf_max = -1, int nb_max = -1, int* host_median_done = nullptr) {
  if (host_median_done) *host_median_done = 0;
  const bool with_stats = stats != nullptr;
  if (M < 0 || C < 0 || T < 0 || L <= 0 || H < L || W < L) return MGB_EINVAL;
  const int64_t pitch = image_pitch > 0 ? image_pitch : W;   // row pitch in elements
  if (pitch < W) return MGB_EINVAL;
  if (itemsize != 1 && itemsize != 2 && itemsize != 4 && itemsize != 8) return MGB_EINVAL;
  if (L > 4096) return MGB_EUNSUPPORTED;
  const int64_t n_roi = M * C * T;
  if (n_roi == 0) return MGB_OK;
  if (n_roi > INT32_MAX) return MGB_EUNSUPPORTED;
  if (!image || (!boxes && marker_stride == 0) || (!roi && !with_stats)) return MGB_EINVAL;
  if (with_stats && (!mask_t || !fg || !bg || Tm <= 0 || itemsize != 2)) return MGB_EINVAL;
  if (g_tma_enabled && marker_stride == 0 && with_stats && nf_max >= 0 && nb_max >= 0) {
    // masked-value lists: sums, means and (optionally) medians in the gather (roi_lists.cu)
    const int rc = roi_gather_lists(image, pitch, C, T, H, W, boxes, order, mask_t, Tm, fg, bg, M, L, roi, stats,
                                    want_median, nf_max, nb_max, host_peers, n_peers, st);
    if (rc == MGB_OK && want_median && host_median_done) *host_median_done = 1;
    if (rc != MGB_EALIGN) return rc;
  }
  if (g_tma_enabled && marker_stride == 0) {
    // TMA-staged path (roi_tma.cu); MGB_EALIGN means "not applicable here", fall through.
    const int rc = roi_gather_tma(image, pitch, C, T, H, W, itemsize, boxes, order, mask_t, Tm, fg, bg, M, L, roi, stats,
                                  host_peers, n_peers, st);
    if (rc != MGB_EALIGN) return rc;
  }
  if (n_peers > 0) return MGB_EUNSUPPORTED;   // peer write-out exists only in the staged kernels
  const int unit = itemsize / 2;
  const int Lu = L * (unit ? unit : 1);
  // (Lu > 2: a row of one word has no 32-bit multiply-high magic number for its division)
  const bool word_path = itemsize >= 2 && (Lu % 2 == 0) && Lu > 2 &&
                         ((reinterpret_cast<uintptr_t>(image) & 3u) == 0) &&
                         (!roi || (reinterpret_cast<uintptr_t>(roi) & 3u) == 0) &&
                         (!with_stats || ((reinterpret_cast<uintptr_t>(fg) & 1u) == 0 &&
                                          (reinterpret_cast<uintptr_t>(bg) & 1u) == 0));
  if (word_path) {
    GatherParams p{};
    p.image = (const uint16_t*)image; p.roi = (uint16_t*)roi;
    p.C = C; p.T = T; p.H = H; p.W = pitch * unit; p.boxes = boxes; p.marker_stride = marker_stride * unit;
    p.unit = unit; p.L = L; p.Lu = Lu;
    p.half = (uint32_t)(Lu / 2); p.magic = magic_for(p.half); p.words = (uint32_t)L * p.half;
    p.mask_t = mask_t; p.Tm = Tm; p.fg = fg; p.bg = bg; p.stats = stats;
    if (with_stats) roi_gather_words_kernel<true><<<(unsigned)n_roi, kThreads, 0, st>>>(p);
    else roi_gather_words_kernel<false><<<(unsigned)n_roi, kThreads, 0, st>>>(p);
  } else if (with_stats) {
    roi_gather_scalar_kernel<uint16_t, true><<<(unsigned)n_roi, kThreads, 0, st>>>(
        (const uint16_t*)image, (uint16_t*)roi, C, T, H, pitch, boxes, marker_stride, L, mask_t, Tm, fg, bg, stats);
  } else {
    switch (itemsize) {
      case 1: roi_gather_scalar_kernel<uint8_t, false><<<(unsigned)n_roi, kThreads, 0, st>>>((const uint8_t*)image, (uint8_t*)roi, C, T, H, pitch, boxes, marker_stride, L, nullptr, 0, nullptr, nullptr, nullptr); break;
      case 2: roi_gather_scalar_kernel<uint16_t, false><<<(unsigned)n_roi, kThreads, 0, st>>>((const uint16_t*)image, (uint16_t*)roi, C, T, H, pitch, boxes, marker_stride, L, nullptr, 0, nullptr, nullptr, nullptr); break;
      case 4: roi_gather_scalar_kernel<uint32_t, false><<<(unsigned)n_roi, kThreads, 0, st>>>((const uint32_t*)image, (uint32_t*)roi, C, T, H, pitch, boxes, marker_stride, L, nullptr, 0, nullptr, nullptr, nullptr); break;
      default: roi_gather_scalar_kernel<uint64_t, false><<<(unsigned)n_roi, kThreads, 0, st>>>((const uint64_t*)image, (uint64_t*)roi, C, T, H, pitch, boxes, marker_stride, L, nullptr, 0, nullptr, nullptr, nullptr); break;
    }
  }
  MGB_CUDA_LAUNCH_CHECK();
  return MGB_OK;
}

int mgb_set_tma_enabled(int enabled) {
  const int old = g_tma_enabled;
  g_tma_enabled = enabled ? 1 : 0;
  return old;
}

int mgb_set_gather_loader(int loader) {
  // bit 0: loader (0 TMA, 1 cp.async); value 2/3 additionally disables the warp-per-marker kernel
  const int old = g_gather_loader | (g_gather_wpm ? 0 : 2);
  if (loader >= 0 && loader <= 3) {
    g_gather_loader = loader & 1;
    g_gather_wpm = (loader & 2) ? 0 : 1;
  }
  return old;
}

int mgb_roi_gather(const void* image, int64_t image_pitch, int64_t C, int64_t T, int64_t H, int64_t W,
                   int itemsize, const int32_t* boxes, const int32_t* order, int64_t M, int L, void* roi,
                   void* stream) {
  if (!roi && M * C * T > 0) return MGB_EINVAL;
  return gather_common(image, image_pitch, C, T, H, W, itemsize, boxes, order, 0, nullptr, 0, nullptr, nullptr, M, L, roi,
                       nullptr, (cudaStream_t)stream);
}

int mgb_roi_gather_stats_u16(const uint16_t* image, int64_t image_pitch, int64_t C, int64_t T, int64_t H,
                             int64_t W, const int32_t* boxes, const int32_t* order, const int32_t* mask_t, int64_t Tm,
                             const uint8_t* fg, const uint8_t* bg, int64_t M, int L,
                             uint16_t* roi, double* stats, int want_median, int fg_count_max, int bg_count_max,
                             int* host_median_done, void* stream) {
  if (host_median_done) *host_median_done = 0;
  if (!stats && M * C * T > 0) return MGB_EINVAL;
  return gather_common(image, image_pitch, C, T, H, W, 2, boxes, order, 0, mask_t, Tm, fg, bg, M, L, roi, stats,
                       (cudaStream_t)stream, nullptr, 0, want_median, fg_count_max, bg_count_max, host_median_done);
}

int mgb_roi_gather_stats_peers_u16(const uint16_t* image, int64_t image_pitch, int64_t C, int64_t T, int64_t H,
                                   int64_t W, const int32_t* boxes, const int32_t* order, const int32_t* mask_t,
                                   int64_t Tm, const uint8_t* fg, const uint8_t* bg, int64_t M, int L,
                                   uint16_t* roi, const uint64_t* host_peer_stats, int n_peers, int want_median,
                                   int fg_count_max, int bg_count_max, int* host_median_done, void* stream) {
  if (host_median_done) *host_median_done = 0;
  if (!host_peer_stats || n_peers < 1 || n_peers > 8) return MGB_EINVAL;
  if (M * C * T == 0) return MGB_OK;
  // `stats` only flags "with summaries" here; every record is written through the peer pointers
  return gather_common(image, image_pitch, C, T, H, W, 2, boxes, order, 0, mask_t, Tm, fg, bg, M, L, roi,
                       reinterpret_cast<double*>(host_peer_stats[0]), (cudaStream_t)stream, host_peer_stats, n_peers,
                       want_median, fg_count_max, bg_count_max, host_median_done);
}

int mgb_roi_stats_u16(const uint16_t* roi, int64_t M, int64_t C, int64_t T, int L, const int32_t* mask_t,
                      int64_t Tm, const uint8_t* fg, const uint8_t* bg, double* stats, void* stream) {
  if (!stats && M * C * T > 0) return MGB_EINVAL;
  // every marker's roi block (C,T,L,L) is read as its own little image with the box at the origin
  return gather_common(roi, 0, C, T, L, L, 2, nullptr, nullptr, C * T * (int64_t)L * L, mask_t, Tm, fg, bg, M, L, nullptr,
                       stats, (cudaStream_t)stream);
}

int mgb_roi_median_u16(const uint16_t* roi, int64_t M, int64_t C, int64_t T, int L,
                       const int32_t* mask_t, int64_t Tm, const uint8_t* mask, double* median,
                       int64_t median_stride, void* stream) {
  return launch_roi_median<uint16_t>(roi, M, C, T, L, mask_t, Tm, mask, median, median_stride, stream);
}

int mgb_roi_median_f32(const float* roi, int64_t M, int64_t C, int64_t T, int L, const int32_t* mask_t, int64_t Tm,
                       const uint8_t* mask, double* median, int64_t median_stride, void* stream) {
  return launch_roi_median<float>(roi, M, C, T, L, mask_t, Tm, mask, median, median_stride, stream);
}

int mgb_roi_stats_f32(const float* roi, int64_t M, int64_t C, int64_t T, int L, const int32_t* mask_t, int64_t Tm,
                      const uint8_t* fg, const uint8_t* bg, double* stats, void* stream) {
  if (M < 0 || C < 0 || T < 0 || L <= 0) return MGB_EINVAL;
  const int64_t n_roi = M * C * T;
  if (n_roi == 0) return MGB_OK;
  if (n_roi > INT32_MAX) return MGB_EUNSUPPORTED;
  if (!roi || !mask_t || !fg || !bg || !stats || Tm <= 0) return MGB_EINVAL;
  roi_stats_f32_kernel<<<(unsigned)n_roi, kThreads, 0, (cudaStream_t)stream>>>(roi, C, T, L, mask_t, Tm, fg, bg, stats);
  MGB_CUDA_LAUNCH_CHECK();
  return MGB_OK;
}

}  // extern "C"
