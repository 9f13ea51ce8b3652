// F1 + F2: flat-field correction (src/magnify/preprocess.py:83-87) and tile stitching
// (src/magnify/stitch.py:22-39), hand-written for sm_100a.
//
// Data layout in HBM: tiles (C,T,R,Cc,H,W) and image (C,T,Him,Wim) row-major.  All kernels are
// HBM-bound streaming kernels: every thread owns one 16-byte vector of a tile row for the whole
// launch and walks over the tiles that share its flat/dark position, so the float64
// coefficients live in registers and each tile byte is read exactly once per pass.
#include <cstdlib>

#include "common.cuh"
#include "ff_core.cuh"

namespace mgb {

// ------------------------------------------------------------------------------------------
// Pass 1a: per-position max of raw uint16 over the planes sharing a table.
// grid = (HW/8/256, K, splits); tiles viewed as (C, P, HW).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 vmax_u16x8(uint4 a, uint4 b) {
  return make_uint4(__vmaxu2(a.x, b.x), __vmaxu2(a.y, b.y), __vmaxu2(a.z, b.z),
                    __vmaxu2(a.w, b.w));
}

constexpr int kTileMaxUnroll = 8;

__global__ void __launch_bounds__(kThreads)
ff_tilemax_u16_kernel(const uint4* __restrict__ tiles, int64_t C, int64_t P, int64_t HW8, int K,
                      int splits, uint4* __restrict__ xmax_partial) {
  const int64_t v = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (v >= HW8) return;
  const int k = blockIdx.y;
  const int s = blockIdx.z;
  // Planes of table k: channel k only (K == C) or every channel (K == 1).
  const int64_t n_planes = (K == 1) ? C * P : P;
  const int64_t first = (K == 1) ? 0 : (int64_t)k * P;
  const int64_t lo = first + n_planes * s / splits;
  const int64_t hi = first + n_planes * (s + 1) / splits;
  uint4 m = make_uint4(0, 0, 0, 0);
  const uint4* p = tiles + lo * HW8 + v;
  int64_t n = hi - lo;
  while (n >= kTileMaxUnroll) {
    uint4 r[kTileMaxUnroll];
#pragma unroll
    for (int j = 0; j < kTileMaxUnroll; ++j) r[j] = ldg_stream(p + (int64_t)j * HW8);
#pragma unroll
    for (int j = 0; j < kTileMaxUnroll; ++j) m = vmax_u16x8(m, r[j]);
    p += (int64_t)kTileMaxUnroll * HW8;
    n -= kTileMaxUnroll;
  }
  for (; n > 0; --n, p += HW8) m = vmax_u16x8(m, ldg_stream(p));
  xmax_partial[((int64_t)s * K + k) * HW8 + v] = m;
}

// ------------------------------------------------------------------------------------------
// Pass 1b: (M, M2) from the per-position maxima, exact float64.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double block_max(double v, double* smem) {
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) smem[w] = v;
  __syncthreads();
  if (w == 0) {
    v = (l < (blockDim.x >> 5)) ? smem[l] : 0.0;
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  }
  __syncthreads();
  return v;
}

// One pixel: t = max(x - dark, 0) and u = t / flat in the reference's operation order, folded into
// the running maxima m1 of t and m2 of u.  xarray's max skips NaN (preprocess.py:84,86); fmax does
// the same.
__device__ __forceinline__ void ff_maxima_step(double x, double dark, double flat, double& m1, double& m2) {
  double t = __dsub_rn(x, dark);
  t = t < 0.0 ? 0.0 : t;
  const double u = __ddiv_rn(t, flat);
  m1 = fmax(m1, t);
  m2 = fmax(m2, u);
}

// The block's maxima folded into maxima[0] (t) and maxima[1] (u).
__device__ __forceinline__ void ff_maxima_finish(double m1, double m2, double* maxima) {
  __shared__ double sm[2][kThreads / 32];
  m1 = block_max(m1, sm[0]);
  m2 = block_max(m2, sm[1]);
  if (threadIdx.x == 0) {
    atomic_max_nonneg_f64(&maxima[0], m1);
    atomic_max_nonneg_f64(&maxima[1], m2);
  }
}

__global__ void __launch_bounds__(kThreads)
ff_maxima_kernel(const uint16_t* __restrict__ xmax_partial, int splits, int K, int64_t HW,
                 const double* __restrict__ flat, const double* __restrict__ dark,
                 double* __restrict__ maxima) {
  double m1 = 0.0, m2 = 0.0;
  const int64_t total = (int64_t)K * HW;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    unsigned x = 0;
    for (int s = 0; s < splits; ++s) x = max(x, (unsigned)xmax_partial[(int64_t)s * total + i]);
    ff_maxima_step((double)x, dark[i], flat[i], m1, m2);
  }
  ff_maxima_finish(m1, m2, maxima);
}

template <typename T>
__global__ void __launch_bounds__(kThreads)
ff_maxima_generic_kernel(const T* __restrict__ tiles, int64_t C, int64_t P, int64_t HW, int K,
                         const double* __restrict__ flat, const double* __restrict__ dark,
                         double* __restrict__ maxima) {
  double m1 = 0.0, m2 = 0.0;
  const int64_t total = C * P * HW;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t pos = i % HW;
    const int64_t k = (K == 1) ? 0 : i / (P * HW);
    ff_maxima_step((double)tiles[i], dark[k * HW + pos], flat[k * HW + pos], m1, m2);
  }
  ff_maxima_finish(m1, m2, maxima);
}

// ------------------------------------------------------------------------------------------
// Pass 2 preparation.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads)
ff_tables_kernel(const double* __restrict__ flat, const double* __restrict__ dark, int64_t n,
                 const double* __restrict__ maxima, double* __restrict__ gain,
                 double* __restrict__ bias) {
  const double M = maxima[0], M2 = maxima[1];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    double g, b;
    ff_make_coeffs(flat[i], dark[i], M, M2, &g, &b);
    gain[i] = g;
    bias[i] = b;
  }
}

// ------------------------------------------------------------------------------------------
// Pass 2: flat-field apply fused with stitch (MODE 1) or plain stitch (MODE 0), 16-bit units.
//
// A thread owns the 8 output pixels xk0..xk0+7 of kept row y (xk = x - clip) for every tile
// whose column cc satisfies cc % P == q; for those tiles cc*w % 8 is the same, so the 16-byte
// output vector is aligned for all of them and the misalignment S of the input (two aligned
// 16-byte loads, funnel-shifted) is a launch constant of the (q) slice.
// ------------------------------------------------------------------------------------------
struct StitchParams {
  const uint16_t* tiles;
  uint16_t* image;
  int64_t CT;      // C*T images
  int T;           // timepoints per channel (table index = ct / T when K > 1)
  int R, Cc;       // tile grid
  int H, W;        // tile size (16-bit units along x)
  int clip;        // first kept pixel (16-bit units along x), rows use clip_y
  int clip_y;
  int h, w;        // kept rows / kept 16-bit units per tile
  int64_t Wim;     // image row pitch in 16-bit units (>= Cc * w; padded so that rows are 16-byte aligned)
  int64_t Him;     // R * h
  int P;           // tile-column period of the output phase
  int K;           // number of coefficient tables (1 or C)
  int ct_splits;   // CTAs sharing one (row, x-block, q, k)
  int xblocks;     // ceil((w + 7) / 8 / 256)
  const double* gain;
  const double* bias;
  const double* flat;
  const double* dark;
  const double* maxima;
};

// Prefetch ring: every thread streams its own aligned 16-byte input chunk of the next
// kStitchStages tiles into shared memory with cp.async (LDGSTS, L1 bypass), so the bytes in
// flight per SM are decoupled from the register file, which holds the 16 float64 coefficients.
// A thread reads back its own slot and (for a shifted vector) its right neighbour's, which
// needs only warp-level synchronisation; every input byte is requested from L2 once.
constexpr int stitch_smem_bytes(int stages) { return stages * (kThreads + kThreads / 32) * 16; }

template <int MODE, int S, int kStitchStages>
__device__ __forceinline__ void stitch_u16_body(const StitchParams& p, uint4* ring, int q, int k, int split) {
  const int bx = blockIdx.x / p.P;              // (row, x-block); the phase slice q varies fastest
  const int xb = bx % p.xblocks;
  const int y = bx / p.xblocks;

  const int phase = (int)(((int64_t)q * p.w) & 7);
  const int j = xb * kThreads + threadIdx.x;   // output vector index within the kept row
  const int xk0 = 8 * j - phase;               // first kept pixel of this thread
  // a warp whose first vector is already right of the kept row has nothing to do (the last
  // active lane of the previous warp streams its own extra chunk)
  if (8 * (j - (int)(threadIdx.x & 31)) - phase >= p.w) return;
  const bool active = xk0 < p.w;               // lanes right of the kept row only feed neighbours
  const int xin0 = p.clip + xk0;               // may be negative for the first vector
  const int a0 = (xin0 - S) >> 3;              // aligned input chunk (exact: xin0 - S = 8 * a0)
  const int chunks = p.W >> 3;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // Every thread streams ONE aligned 16-byte chunk per tile; the second chunk a shifted vector
  // needs (S != 0) is the next lane's chunk, read back from its ring slot after a __syncwarp.
  // Lane 31 has no next lane in its warp, so it also streams chunk a0+1 into a per-warp slot.
  const bool ld_a = (a0 >= 0) && (a0 < chunks);
  const bool ld_x = (S != 0) && (lane == 31) && (a0 + 1 >= 0) && (a0 + 1 < chunks);
  const bool full = active && (xk0 >= 0) && (xk0 + 8 <= p.w);

  // Images handled by this CTA: table k covers ct in [k*T, (k+1)*T) when K > 1.
  const int64_t n_ct = (p.K == 1) ? p.CT : p.T;
  const int64_t ct_first = (p.K == 1) ? 0 : (int64_t)k * p.T;
  const int64_t ct_lo = ct_first + n_ct * split / p.ct_splits;
  const int64_t ct_hi = ct_first + n_ct * (split + 1) / p.ct_splits;
  const int cols_q = (p.Cc - q + p.P - 1) / p.P;   // tile columns q, q+P, ...
  const int n_iter = (int)((ct_hi - ct_lo) * p.R * cols_q);   // host keeps this below 2^31
  if (n_iter <= 0) return;

  // Tiles are visited in (ct, r, cc) order, cc fastest with stride P.  Between consecutive
  // tiles both offsets advance by a constant, except every cols_q-th step (next tile row; the
  // step from the last tile row of an image to the next image is the same).
  const int64_t tile_stride = (int64_t)p.H * p.W;
  const int64_t in_step = (int64_t)p.P * tile_stride;
  const int64_t in_wrap = (int64_t)(p.Cc - (cols_q - 1) * p.P) * tile_stride;
  const int64_t in_step8 = in_step >> 3, in_wrap8 = in_wrap >> 3;   // in 16-byte vectors
  const int64_t out_step = (int64_t)p.P * p.w;
  const int64_t out_wrap = (int64_t)p.h * p.Wim - (int64_t)(cols_q - 1) * p.P * p.w;
  const uint4* ip = reinterpret_cast<const uint4*>(
                        p.tiles + ((ct_lo * p.R * p.Cc + q) * tile_stride + (int64_t)(p.clip_y + y) * p.W)) + a0;
  uint16_t* op = p.image + ((ct_lo * p.Him + y) * p.Wim + (int64_t)q * p.w + xk0);
  int ci_in = 0, ci_out = 0;

  constexpr int kStageVecs = kThreads + kThreads / 32;       // 256 chunks + one spare per warp
  uint4* slot_a = ring + threadIdx.x;
  uint4* slot_b = (lane < 31) ? slot_a + 1 : ring + kThreads + warp;
  const uint32_t sa = (uint32_t)__cvta_generic_to_shared(slot_a);
  const uint32_t sx = (uint32_t)__cvta_generic_to_shared(ring + kThreads + warp);
  if (!ld_a) {
#pragma unroll
    for (int s = 0; s < kStitchStages; ++s) slot_a[s * kStageVecs] = make_uint4(0, 0, 0, 0);
  }
  if (S != 0 && lane == 31 && !ld_x) {
#pragma unroll
    for (int s = 0; s < kStitchStages; ++s) ring[s * kStageVecs + kThreads + warp] = make_uint4(0, 0, 0, 0);
  }

  auto issue = [&](int stage) {
    if (ld_a) cp_async16(sa + stage * (kStageVecs * 16), ip);
    if (ld_x) cp_async16(sx + stage * (kStageVecs * 16), ip + 1);
    const bool wrap = (++ci_in == cols_q);
    if (wrap) ci_in = 0;
    ip += wrap ? in_wrap8 : in_step8;
  };

  // prologue: kStitchStages-1 tiles in flight
#pragma unroll
  for (int s = 0; s < kStitchStages - 1; ++s) {
    if (s < n_iter) issue(s);
    cp_async_commit();
  }
  // coefficient loads are issued after the ring prologue so that both are in flight together
  double g[8], b[8];
  if constexpr (MODE == 1) {
    const int64_t base = ((int64_t)k * p.H + (p.clip_y + y)) * p.W;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int xi = xin0 + i;
      const bool in = active && (xi >= 0) && (xi < p.W);
      // out-of-row lanes: s = 2^20 + 2^19 + 0.5 never trips the guard (their result is not stored)
      g[i] = in ? p.gain[base + xi] : 0.0;
      b[i] = in ? p.bias[base + xi] : 1572864.5;
    }
  }

  int stage = 0;
  for (int it = 0; it < n_iter; ++it) {
    // refill the stage consumed in the previous iteration (all lanes are past reading it), then
    // wait for this iteration's chunk -- and, for a shifted vector, the neighbours' chunks
    if constexpr (S != 0) __syncwarp();
    if (it + kStitchStages - 1 < n_iter) {
      int pf = stage + kStitchStages - 1;
      if (pf >= kStitchStages) pf -= kStitchStages;
      issue(pf);
    }
    cp_async_commit();
    cp_async_wait<kStitchStages - 1>();
    if constexpr (S != 0) __syncwarp();
    const uint4 va = slot_a[stage * kStageVecs];
    const uint4 vb = (S != 0) ? slot_b[stage * kStageVecs] : va;
    if (++stage == kStitchStages) stage = 0;

    uint4 v = shift_units<S>(va, vb);
    if constexpr (MODE == 1) {
      const uint32_t win[4] = {v.x, v.y, v.z, v.w};
      uint32_t wout[4];
      bool slow = false;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int o0 = ff_fast_px(__byte_perm(win[i], kFFHiBase, 0x7610), g[2 * i], b[2 * i], &slow);
        const int o1 = ff_fast_px(__byte_perm(win[i], kFFHiBase, 0x7632), g[2 * i + 1], b[2 * i + 1], &slow);
        wout[i] = __byte_perm((uint32_t)o0, (uint32_t)o1, 0x5410);
      }
      if (slow) {
        // Rare: some pixel is within 2^-24 of an integer (or has unusable coefficients).
        // Recompute the whole vector in the reference's exact operation order.
        const double M = p.maxima[0], M2 = p.maxima[1];
        const int64_t base = ((int64_t)k * p.H + (p.clip_y + y)) * p.W;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int xi = xin0 + i;
          if (xi < 0 || xi >= p.W) continue;
          const uint16_t x = (uint16_t)((win[i >> 1] >> (16 * (i & 1))) & 0xffffu);
          const uint16_t e = ff_exact_u16(x, p.flat[base + xi], p.dark[base + xi], M, M2);
          wout[i >> 1] = (i & 1) ? ((wout[i >> 1] & 0x0000ffffu) | ((uint32_t)e << 16))
                                 : ((wout[i >> 1] & 0xffff0000u) | (uint32_t)e);
        }
      }
      v = make_uint4(wout[0], wout[1], wout[2], wout[3]);
    }
    if (full) {
      stg_stream(reinterpret_cast<uint4*>(op), v);
    } else {
      const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int xk = xk0 + i;
        if (xk >= 0 && xk < p.w) op[i] = (uint16_t)((wv[i >> 1] >> (16 * (i & 1))) & 0xffffu);
      }
    }
    const bool owrap = (++ci_out == cols_q);
    if (owrap) ci_out = 0;
    op += owrap ? out_wrap : out_step;
  }
}

// One launch covers every output phase.  The phase slice q is the fastest-varying block index, so
// the CTAs that write the adjacent column segments of one image row are co-resident and the
// partially written 128-byte lines at the segment boundaries merge in L2 instead of costing a
// DRAM read-modify-write each.  The input shift S is uniform per CTA: the tile loop is
// instantiated once per S and selected with a CTA-uniform switch.
template <int MODE, int kStitchStages, int kMinBlocks>
__global__ void __launch_bounds__(kThreads, kMinBlocks) stitch_u16_kernel(const StitchParams p) {
  extern __shared__ uint4 ring[];   // [stage][2][kThreads]
  const int q = blockIdx.x % p.P;
  const int k = blockIdx.y;
  const int split = blockIdx.z;
  const int phase = (int)(((int64_t)q * p.w) & 7);
  const int S = (((p.clip - phase) % 8) + 8) % 8;
  switch (S) {
    case 0: stitch_u16_body<MODE, 0, kStitchStages>(p, ring, q, k, split); break;
    case 1: stitch_u16_body<MODE, 1, kStitchStages>(p, ring, q, k, split); break;
    case 2: stitch_u16_body<MODE, 2, kStitchStages>(p, ring, q, k, split); break;
    case 3: stitch_u16_body<MODE, 3, kStitchStages>(p, ring, q, k, split); break;
    case 4: stitch_u16_body<MODE, 4, kStitchStages>(p, ring, q, k, split); break;
    case 5: stitch_u16_body<MODE, 5, kStitchStages>(p, ring, q, k, split); break;
    case 6: stitch_u16_body<MODE, 6, kStitchStages>(p, ring, q, k, split); break;
    default: stitch_u16_body<MODE, 7, kStitchStages>(p, ring, q, k, split); break;
  }
}

// Element-wise fallbacks (any itemsize / any shape).
template <typename T>
__global__ void __launch_bounds__(kThreads)
stitch_generic_kernel(const T* __restrict__ tiles, T* __restrict__ image, int64_t CT, int R, int Cc,
                      int H, int W, int clip, int h, int w, int64_t pitch) {
  const int64_t Wim = (int64_t)Cc * w, Him = (int64_t)R * h;
  const int64_t total = CT * Him * Wim;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t X = i % Wim;
    const int64_t Y = (i / Wim) % Him;
    const int64_t ct = i / (Wim * Him);
    const int cc = (int)(X / w), x = (int)(X % w);
    const int r = (int)(Y / h), y = (int)(Y % h);
    image[(ct * Him + Y) * pitch + X] = tiles[(((ct * R + r) * Cc + cc) * H + clip + y) * (int64_t)W + clip + x];
  }
}

template <typename T>
__device__ __forceinline__ T ff_cast(double v);
template <> __device__ __forceinline__ uint8_t ff_cast<uint8_t>(double v) { return (uint8_t)(long long)v; }
template <> __device__ __forceinline__ uint16_t ff_cast<uint16_t>(double v) { return (uint16_t)(long long)v; }
template <> __device__ __forceinline__ float ff_cast<float>(double v) { return __double2float_rn(v); }
template <> __device__ __forceinline__ double ff_cast<double>(double v) { return v; }

template <typename T>
__global__ void __launch_bounds__(kThreads)
ff_apply_generic_kernel(const T* __restrict__ tiles, T* __restrict__ out, int64_t C, int64_t P,
                        int64_t HW, int K, const double* __restrict__ flat,
                        const double* __restrict__ dark, const double* __restrict__ maxima) {
  const double M = maxima[0], M2 = maxima[1];
  const int64_t total = C * P * HW;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t pos = i % HW;
    const int64_t k = (K == 1) ? 0 : i / (P * HW);
    out[i] = ff_cast<T>(ff_exact_value((double)tiles[i], flat[k * HW + pos], dark[k * HW + pos], M, M2));
  }
}

static int g_stitch_variant = 0;   // tuning knob: 0 = 6 stages x 2 CTAs/SM, 1 = 11 x 2, 2 = 8 x 3

template <int MODE, int D, int B>
static int launch_stitch_variant(const StitchParams& p, cudaStream_t st) {
  dim3 grid((unsigned)(p.h * p.xblocks * p.P), (unsigned)p.K, (unsigned)p.ct_splits);
  constexpr int smem = stitch_smem_bytes(D);
  static bool attr_set = false;
  if (!attr_set && smem > 48 * 1024) {
    MGB_CUDA_TRY(cudaFuncSetAttribute(stitch_u16_kernel<MODE, D, B>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_set = true;
  }
  stitch_u16_kernel<MODE, D, B><<<grid, kThreads, smem, st>>>(p);
  MGB_CUDA_LAUNCH_CHECK();
  return MGB_OK;
}

template <int MODE>
static int launch_stitch_fast(const StitchParams& p, cudaStream_t st) {
  switch (g_stitch_variant) {
    case 1: return launch_stitch_variant<MODE, 11, 2>(p, st);
    case 2: return launch_stitch_variant<MODE, 8, 3>(p, st);
    default: return launch_stitch_variant<MODE, 6, 2>(p, st);
  }
}

static int gcd_int(int a, int b) { while (b) { int t = a % b; a = b; b = t; } return a; }

static int cached_sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
  }
  return n;
}

// Launch the vectorised stitch (MODE 0) / flat-field+stitch (MODE 1) over 16-bit units.
// The output phase of tile column cc is (cc * w) mod 8 and repeats with period P, so the
// columns are processed in P slices, each with its own compile-time input shift S.
template <int MODE>
static int run_stitch_fast(StitchParams p, cudaStream_t st) {
  const int wm = p.w & 7;
  p.P = wm ? 8 / gcd_int(wm, 8) : 1;
  if (p.P > p.Cc) p.P = p.Cc;
  p.xblocks = (int)ceil_div(ceil_div((int64_t)p.w + 7, 8), kThreads);
  // Enough CTAs for several waves at 2 CTAs/SM without shortening the per-thread tile loop
  // below ~16 iterations (the register-resident coefficients are loaded once per CTA).
  const int64_t base_ctas = (int64_t)p.h * p.xblocks * p.K * p.P;
  const int64_t n_ct = (p.K == 1) ? p.CT : p.T;
  const int64_t cols_q = (p.Cc + p.P - 1) / p.P;
  if (n_ct * p.R * cols_q >= INT32_MAX) return MGB_EUNSUPPORTED;   // 32-bit tile loop counter
  // Split the tile loop over images so that (a) there are enough CTAs for several waves and (b) a
  // CTA walks ~kTargetIters tiles: blockIdx.z is the slowest grid index, so the resident CTAs all
  // work on the same narrow band of tiles (DRAM page locality; long loops let CTAs drift apart and
  // measured 15-20% slower), while the register-resident coefficients are still amortised.
  int64_t target_iters = MODE == 1 ? 160 : 32;   // the copy-only kernel has no coefficients to amortise
  if (const char* e = getenv("MGB_STITCH_ITERS")) target_iters = atoll(e) > 0 ? atoll(e) : target_iters;  // tuning
  const int64_t iters_per_ct = p.R * cols_q;
  int64_t splits = (n_ct * iters_per_ct + target_iters - 1) / target_iters;
  while (base_ctas * splits < (int64_t)cached_sm_count() * 16 && (n_ct / (splits + 1)) * iters_per_ct >= 16) ++splits;
  if (splits > n_ct) splits = n_ct;
  if (splits > 32768) splits = 32768;
  if (splits < 1) splits = 1;
  p.ct_splits = (int)splits;
  if (p.K > 65535 || splits > 65535 || (int64_t)p.h * p.xblocks * p.P > INT32_MAX) return MGB_EUNSUPPORTED;
  return launch_stitch_fast<MODE>(p, st);
}

// The checks both stitch entry points make, and the geometry of p in 16-bit units (`units` per
// element along x; rows stay in elements).  An empty stack returns MGB_OK with p->CT == 0: nothing
// to launch.  K (tables) counts toward the size limits, tables_ok (no table pointer is null) toward
// the pointer check.  limits_first puts the size limits before the empty-stack shortcut and the
// null pointers (mgb_stitch), else after them (mgb_flatfield_stitch_u16): an empty stack of too tall
// tiles is MGB_EUNSUPPORTED for one entry point and MGB_OK for the other.
static int stitch_setup(const void* tiles, void* image, int64_t image_pitch, int64_t C, int64_t T, int64_t R,
                        int64_t Cc, int64_t H, int64_t W, int64_t overlap, int units, int K, bool tables_ok,
                        bool limits_first, StitchParams* p) {
  *p = StitchParams{};
  if (C < 0 || T < 0 || R < 0 || Cc < 0 || H <= 0 || W <= 0) return MGB_EINVAL;
  if (overlap < 0 || overlap >= H || overlap >= W) return MGB_EINVAL;  // stitch.py:8-9,16-20
  const bool too_large = H > INT32_MAX / 8 || W > INT32_MAX / 8 || R > INT32_MAX || Cc > INT32_MAX || K > 65535;
  if (limits_first && too_large) return MGB_EUNSUPPORTED;
  if (C * T == 0 || R == 0 || Cc == 0) return MGB_OK;
  if (!tiles || !image || !tables_ok) return MGB_EINVAL;
  if (too_large) return MGB_EUNSUPPORTED;
  const int clip = (int)(overlap / 2);
  const int h = (int)(H - overlap), w = (int)(W - overlap);
  const int64_t pitch = image_pitch > 0 ? image_pitch : Cc * w;
  if (pitch < Cc * w) return MGB_EINVAL;
  p->tiles = (const uint16_t*)tiles; p->image = (uint16_t*)image;
  p->CT = C * T; p->T = (int)T; p->R = (int)R; p->Cc = (int)Cc;
  p->H = (int)H; p->W = (int)(W * units); p->clip = clip * units; p->clip_y = clip; p->h = h; p->w = w * units;
  p->Wim = pitch * units; p->Him = R * h; p->K = K;
  return MGB_OK;
}

// The vectorised kernels read and write whole 16-byte vectors.
static bool stitch_vectorisable(const StitchParams& p) {
  return p.W % 8 == 0 && p.Wim % 8 == 0 && aligned16(p.tiles) && aligned16(p.image);
}

static int grid_for(int64_t n) {
  int64_t b = ceil_div(n, kThreads);
  const int64_t cap = (int64_t)cached_sm_count() * 32;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

}  // namespace mgb

using namespace mgb;

extern "C" {

int mgb_sm_count(void) { return cached_sm_count(); }

int mgb_set_stitch_variant(int variant) {
  const int old = g_stitch_variant;
  if (variant >= 0 && variant <= 2) g_stitch_variant = variant;
  return old;
}

int mgb_stitch(const void* tiles, void* image, int64_t image_pitch, int64_t C, int64_t T, int64_t R,
               int64_t Cc, int64_t H, int64_t W, int64_t overlap, int itemsize, int* host_used_fast,
               void* stream) {
  if (host_used_fast) *host_used_fast = 0;
  if (itemsize != 1 && itemsize != 2 && itemsize != 4 && itemsize != 8) return MGB_EINVAL;
  // 16-bit units per element; bytes (element-wise kernel only) keep the geometry in elements
  const int u = itemsize >= 2 ? itemsize / 2 : 1;
  StitchParams p;
  const int rc = stitch_setup(tiles, image, image_pitch, C, T, R, Cc, H, W, overlap, u, /*K=*/1,
                              /*tables_ok=*/true, /*limits_first=*/true, &p);
  if (rc != MGB_OK || p.CT == 0) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (itemsize >= 2 && stitch_vectorisable(p)) {
    if (host_used_fast) *host_used_fast = 1;
    return run_stitch_fast<0>(p, st);
  }
  // the element-wise kernel takes the geometry in elements
  const int We = p.W / u, w = p.w / u;
  const int64_t pitch = p.Wim / u;
  const int64_t total = p.CT * p.Him * p.Cc * w;
  const int g = grid_for(total);
  switch (itemsize) {
    case 1: stitch_generic_kernel<uint8_t><<<g, kThreads, 0, st>>>((const uint8_t*)tiles, (uint8_t*)image, p.CT, p.R, p.Cc, p.H, We, p.clip_y, p.h, w, pitch); break;
    case 2: stitch_generic_kernel<uint16_t><<<g, kThreads, 0, st>>>((const uint16_t*)tiles, (uint16_t*)image, p.CT, p.R, p.Cc, p.H, We, p.clip_y, p.h, w, pitch); break;
    case 4: stitch_generic_kernel<uint32_t><<<g, kThreads, 0, st>>>((const uint32_t*)tiles, (uint32_t*)image, p.CT, p.R, p.Cc, p.H, We, p.clip_y, p.h, w, pitch); break;
    default: stitch_generic_kernel<uint64_t><<<g, kThreads, 0, st>>>((const uint64_t*)tiles, (uint64_t*)image, p.CT, p.R, p.Cc, p.H, We, p.clip_y, p.h, w, pitch); break;
  }
  MGB_CUDA_LAUNCH_CHECK();
  return MGB_OK;
}

int mgb_flatfield_tilemax_u16(const uint16_t* tiles, int64_t C, int64_t P, int64_t HW, int K,
                              int splits, uint16_t* xmax_partial, void* stream) {
  if (!tiles || !xmax_partial || C <= 0 || P <= 0 || HW <= 0 || splits <= 0) return MGB_EINVAL;
  if (K != 1 && K != C) return MGB_EINVAL;
  if (HW % 8 != 0 || !aligned16(tiles) || !aligned16(xmax_partial)) return MGB_EALIGN;
  if (splits > 65535 || K > 65535) return MGB_EUNSUPPORTED;
  const int64_t HW8 = HW / 8;
  dim3 grid((unsigned)ceil_div(HW8, kThreads), (unsigned)K, (unsigned)splits);
  ff_tilemax_u16_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(
      (const uint4*)tiles, C, P, HW8, K, splits, (uint4*)xmax_partial);
  MGB_CUDA_LAUNCH_CHECK();
  return MGB_OK;
}

int mgb_flatfield_maxima(const uint16_t* xmax_partial, int splits, int K, int64_t HW,
                         const double* flat, const double* dark, double* maxima, void* stream) {
  if (!xmax_partial || !flat || !dark || !maxima || splits <= 0 || K <= 0 || HW <= 0) return MGB_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  ff_maxima_kernel<<<grid_for((int64_t)K * HW), kThreads, 0, st>>>(xmax_partial, splits, K, HW, flat, dark, maxima);
  MGB_CUDA_LAUNCH_CHECK();
  return MGB_OK;
}

int mgb_flatfield_maxima_generic(const void* tiles, int dtype, int64_t C, int64_t P, int64_t HW,
                                 int K, const double* flat, const double* dark, double* maxima,
                                 void* stream) {
  if (!tiles || !flat || !dark || !maxima || C <= 0 || P <= 0 || HW <= 0) return MGB_EINVAL;
  if (K != 1 && K != C) return MGB_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  const int g = grid_for(C * P * HW);
  switch (dtype) {
    case MGB_U8: ff_maxima_generic_kernel<uint8_t><<<g, kThreads, 0, st>>>((const uint8_t*)tiles, C, P, HW, K, flat, dark, maxima); break;
    case MGB_U16: ff_maxima_generic_kernel<uint16_t><<<g, kThreads, 0, st>>>((const uint16_t*)tiles, C, P, HW, K, flat, dark, maxima); break;
    case MGB_F32: ff_maxima_generic_kernel<float><<<g, kThreads, 0, st>>>((const float*)tiles, C, P, HW, K, flat, dark, maxima); break;
    case MGB_F64: ff_maxima_generic_kernel<double><<<g, kThreads, 0, st>>>((const double*)tiles, C, P, HW, K, flat, dark, maxima); break;
    default: return MGB_EUNSUPPORTED;
  }
  MGB_CUDA_LAUNCH_CHECK();
  return MGB_OK;
}

int mgb_flatfield_tables(const double* flat, const double* dark, int K, int64_t HW,
                         const double* maxima, double* gain, double* bias, void* stream) {
  if (!flat || !dark || !maxima || !gain || !bias || K <= 0 || HW <= 0) return MGB_EINVAL;
  ff_tables_kernel<<<grid_for((int64_t)K * HW), kThreads, 0, (cudaStream_t)stream>>>(
      flat, dark, (int64_t)K * HW, maxima, gain, bias);
  MGB_CUDA_LAUNCH_CHECK();
  return MGB_OK;
}

int mgb_flatfield_stitch_u16(const uint16_t* tiles, uint16_t* image, int64_t image_pitch, int64_t C,
                             int64_t T, int64_t R, int64_t Cc, int64_t H, int64_t W, int64_t overlap, int K,
                             const double* flat, const double* dark, const double* gain,
                             const double* bias, const double* maxima, void* stream) {
  if (K != 1 && K != C) return MGB_EINVAL;
  const bool tables_ok = flat && dark && gain && bias && maxima;
  StitchParams p;
  const int rc = stitch_setup(tiles, image, image_pitch, C, T, R, Cc, H, W, overlap, 1, K, tables_ok,
                              /*limits_first=*/false, &p);
  if (rc != MGB_OK || p.CT == 0) return rc;
  if (!stitch_vectorisable(p)) return MGB_EALIGN;
  p.gain = gain; p.bias = bias; p.flat = flat; p.dark = dark; p.maxima = maxima;
  return run_stitch_fast<1>(p, (cudaStream_t)stream);
}

int mgb_flatfield_apply_generic(const void* tiles, void* out, int dtype, int64_t C, int64_t P,
                                int64_t HW, int K, const double* flat, const double* dark,
                                const double* maxima, void* stream) {
  if (!tiles || !out || !flat || !dark || !maxima || C <= 0 || P <= 0 || HW <= 0) return MGB_EINVAL;
  if (K != 1 && K != C) return MGB_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  const int g = grid_for(C * P * HW);
  switch (dtype) {
    case MGB_U8: ff_apply_generic_kernel<uint8_t><<<g, kThreads, 0, st>>>((const uint8_t*)tiles, (uint8_t*)out, C, P, HW, K, flat, dark, maxima); break;
    case MGB_U16: ff_apply_generic_kernel<uint16_t><<<g, kThreads, 0, st>>>((const uint16_t*)tiles, (uint16_t*)out, C, P, HW, K, flat, dark, maxima); break;
    case MGB_F32: ff_apply_generic_kernel<float><<<g, kThreads, 0, st>>>((const float*)tiles, (float*)out, C, P, HW, K, flat, dark, maxima); break;
    case MGB_F64: ff_apply_generic_kernel<double><<<g, kThreads, 0, st>>>((const double*)tiles, (double*)out, C, P, HW, K, flat, dark, maxima); break;
    default: return MGB_EUNSUPPORTED;
  }
  MGB_CUDA_LAUNCH_CHECK();
  return MGB_OK;
}

}  // extern "C"
