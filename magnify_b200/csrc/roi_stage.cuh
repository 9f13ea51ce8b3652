// Shared pieces of the staged ROI-gather kernels (roi_tma.cu, roi_lists.cu): the launch
// parameters, mbarrier / TMA wrappers, the copy loops that re-align a window staged in shared
// memory and store it with aligned vector stores, and the host-side set-up both launchers share.
// The arguments of a gather call (GatherArgs) are filled by the entry points in roi.cu.
#pragma once
#include <cstdlib>
#include <type_traits>

#include <cuda.h>
#include <cudaTypedefs.h>

#include "common.cuh"

namespace mgb {

constexpr int kTmaMaxWarps = 8;

struct TmaGatherParams {
  uint16_t* roi;            // may be null (summaries only)
  const int32_t* boxes;     // (M,T,2) in elements
  const int32_t* order;     // (M) processing order of the markers, or null
  const int32_t* mask_t;    // (T) or null when !stats
  const uint8_t* fg;        // (M,Tm,rows,rows) or null
  const uint8_t* bg;
  double* stats;            // (M,C,T,8) or null
  double* peer_stats[8];    // peer-mapped copies of the gathered (ranks,M,C,T,8) buffer, this rank's block
  int n_peers;              // 0: write only `stats`
  int64_t C, T, Tm;
  int rows;                 // L
  int wu;                   // row length in 16-bit units (L * unit)
  int wpu;                  // TMA box width: roundup8(wu + 7) units
  int unit;                 // 16-bit units per element
  int n_stages;
  int loader;               // 0 = TMA tensor copy, 1 = cp.async chunks (sector granularity)
  const uint16_t* image;    // 16-bit units, for the cp.async loader
  int64_t H, Wu;
  int stage_bytes;          // rows * wpu * 2 rounded up to 128
  uint32_t vpr;             // 16-byte vectors per roi row (wu / 8) when the vector path applies, else 0
  uint32_t magic_vpr;       // ceil(2^32 / vpr)
  uint32_t half;            // wu / 2 words per row when the word path applies, else 0
  uint32_t magic_half;
  uint32_t magic_wu;        // ceil(2^32 / wu)
  // masked-value lists (roi_lists.cu)
  int cap_f, cap_b;         // list capacities (entries), multiples of 32
  int want_median;          // 0: sums / means only
  int store;                // 0: summaries only (roi == null)
  int split_parts;          // CTA layout: CTAs sharing each marker from split_from on (1: none)
  int64_t split_from;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0,
                                            int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// The timepoints whose mask timestep is tm (all of them when !MASKED), listed in tlist by one warp;
// returns their number.
template <bool MASKED>
__device__ __forceinline__ int list_timepoints(const TmaGatherParams& p, int tm, int32_t* tlist, int lane) {
  int n = 0;
  for (int64_t base = 0; base < p.T; base += 32) {
    const int64_t t = base + lane;
    const bool hit = (t < p.T) && (!MASKED || p.mask_t[t] == tm);
    const unsigned bal = __ballot_sync(0xffffffffu, hit);
    if (hit) tlist[n + __popc(bal & ((1u << lane) - 1))] = (int32_t)t;
    n += __popc(bal);
  }
  return n;
}

// Called by lane 0: the warp's n stage barriers (one arrival each), made visible to the TMA unit.
__device__ __forceinline__ void init_stage_barriers(uint64_t* bars, int n) {
  for (int s = 0; s < n; ++s) mbar_init(smem_u32(&bars[s]), 1);
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

// Called by lane 0: arm the stage barrier `bar` for tx_bytes and load window (c, t) of marker m to
// `dst`.  The box starts at the 16-byte boundary at or left of the window (a TMA coordinate must
// be a multiple of 16 bytes); the consumer applies the residual shift of 0..7 units.
__device__ __forceinline__ void load_window(const CUtensorMap* tmap, const TmaGatherParams& p, int unit, int64_t m,
                                            int64_t c, int64_t t, uint32_t dst, uint32_t bar, uint32_t tx_bytes) {
  const int32_t top = p.boxes[(m * p.T + t) * 2];
  const int32_t left = p.boxes[(m * p.T + t) * 2 + 1];
  mbar_expect_tx(bar, tx_bytes);
  tma_load_3d(dst, tmap, bar, (left * unit) & ~7, top, (int)(c * p.T + t));
}

// Summary write-out: one record of kStatsRec doubles per (marker, channel, time) (medians NaN when
// the kernel does not compute them).  With peers, the 64-byte record goes straight into this rank's
// block of the gathered buffer of EVERY rank (NVLink peer stores, one lane per peer): the
// per-marker summaries are all-gathered by the kernel that computes them, no separate collective.
__device__ __forceinline__ void write_stats(const TmaGatherParams& p, int lane, int64_t n, double cf, double cb,
                                            double sf, double sb, double mf, double mb) {
  // called by the whole warp (all lanes hold the reduced values): lane 0 writes the local record,
  // or lane j writes the record to peer j (one 64-byte record = four 16-byte stores per peer)
  double* o = nullptr;
  if (p.n_peers == 0) {
    if (lane == 0) o = p.stats + n * kStatsRec;
  } else if (lane < p.n_peers) {
    o = p.peer_stats[lane] + n * kStatsRec;
  }
  if (o) {
    double2* o2 = reinterpret_cast<double2*>(o);
    o2[0] = make_double2(cf, cb);
    o2[1] = make_double2(sf, sb);
    o2[2] = make_double2(sf / cf, sb / cb);   // 0/0 = NaN like nanmean
    o2[3] = make_double2(mf, mb);
  }
}

// Vector path for one window: rows of wu = 8*vpr units, output 16-byte aligned.
// VPL > 0: the loop over this lane's vectors is fully unrolled and the lane's mask bytes and
// shared-memory offsets (which do not depend on the window) live in registers for the whole CTA.
template <bool STATS, bool STORE, int S, int VPL>
__device__ __forceinline__ void consume_vec(const TmaGatherParams& p, const uint8_t* buf, uint16_t* dst,
                                            const uint8_t* fgm, const uint8_t* bgm, int lane,
                                            const uint2* fm, const uint2* bm, const uint32_t* svo,
                                            uint32_t* sf_out, uint32_t* sb_out) {
  const uint4* s4 = reinterpret_cast<const uint4*>(buf);
  uint4* d4 = reinterpret_cast<uint4*>(dst);
  const uint32_t nvec = p.rows * p.vpr;
  uint32_t sf = 0, sb = 0;
  if constexpr (VPL > 0) {
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
      const uint32_t v = lane + 32 * k;
      if (v < nvec) {
        const uint4 a = s4[svo[k]];
        const uint4 b = (S != 0) ? s4[svo[k] + 1] : a;
        const uint4 d = shift_units<S>(a, b);
        if constexpr (STORE) stg_stream(d4 + v, d);
        if constexpr (STATS) {
          sf = __dp2a_lo(d.x, fm[k].x, sf); sf = __dp2a_hi(d.y, fm[k].x, sf);
          sf = __dp2a_lo(d.z, fm[k].y, sf); sf = __dp2a_hi(d.w, fm[k].y, sf);
          sb = __dp2a_lo(d.x, bm[k].x, sb); sb = __dp2a_hi(d.y, bm[k].x, sb);
          sb = __dp2a_lo(d.z, bm[k].y, sb); sb = __dp2a_hi(d.w, bm[k].y, sb);
        }
      }
    }
  } else {
    const uint2* f2 = reinterpret_cast<const uint2*>(fgm);
    const uint2* b2 = reinterpret_cast<const uint2*>(bgm);
    const uint32_t pitch = p.wpu >> 3;
#pragma unroll 4
    for (uint32_t v = lane; v < nvec; v += 32) {
      const uint32_t row = __umulhi(v, p.magic_vpr);
      const uint32_t sv = row * pitch + (v - row * p.vpr);
      const uint4 a = s4[sv];
      const uint4 b = (S != 0) ? s4[sv + 1] : a;
      const uint4 d = shift_units<S>(a, b);
      if constexpr (STORE) stg_stream(d4 + v, d);
      if constexpr (STATS) {
        const uint2 f = f2[v];
        const uint2 g = b2[v];
        sf = __dp2a_lo(d.x, f.x, sf); sf = __dp2a_hi(d.y, f.x, sf);
        sf = __dp2a_lo(d.z, f.y, sf); sf = __dp2a_hi(d.w, f.y, sf);
        sb = __dp2a_lo(d.x, g.x, sb); sb = __dp2a_hi(d.y, g.x, sb);
        sb = __dp2a_lo(d.z, g.y, sb); sb = __dp2a_hi(d.w, g.y, sb);
      }
    }
  }
  *sf_out = sf;
  *sb_out = sb;
}

// Word / unit path for rows that are not a whole number of 16-byte vectors (e.g. L = 50).
template <bool STATS, bool STORE>
__device__ __forceinline__ void consume_generic(const TmaGatherParams& p, const uint8_t* buf, uint16_t* dst,
                                                const uint8_t* fgm, const uint8_t* bgm, int lane, int shift,
                                                uint32_t* sf_out, uint32_t* sb_out) {
  const uint16_t* s16 = reinterpret_cast<const uint16_t*>(buf);
  uint32_t sf = 0, sb = 0;
  if (p.half) {
    uint32_t* d32 = reinterpret_cast<uint32_t*>(dst);
    const uint16_t* f16 = reinterpret_cast<const uint16_t*>(fgm);
    const uint16_t* b16 = reinterpret_cast<const uint16_t*>(bgm);
    const uint32_t words = p.rows * p.half;
#pragma unroll 4
    for (uint32_t w = lane; w < words; w += 32) {
      const uint32_t row = __umulhi(w, p.magic_half);
      const uint32_t u = row * p.wpu + shift + 2 * (w - row * p.half);
      const uint32_t d = (uint32_t)s16[u] | ((uint32_t)s16[u + 1] << 16);
      if constexpr (STORE) d32[w] = d;
      if constexpr (STATS) {
        sf = __dp2a_lo(d, (uint32_t)f16[w], sf);
        sb = __dp2a_lo(d, (uint32_t)b16[w], sb);
      }
    }
  } else {
    const int total = p.rows * p.wu;
    for (int e = lane; e < total; e += 32) {
      const int row = e / p.wu;
      const uint32_t d = s16[row * p.wpu + shift + (e - row * p.wu)];
      if constexpr (STORE) dst[e] = (uint16_t)d;
      if constexpr (STATS) {
        sf += fgm[e] ? d : 0u;
        sb += bgm[e] ? d : 0u;
      }
    }
  }
  *sf_out = sf;
  *sb_out = sb;
}

template <int PAR>
__device__ __forceinline__ uint32_t load_pair(const uint32_t* s32, uint32_t unit_off) {
  const uint32_t w = unit_off >> 1;
  if constexpr (PAR == 0) {
    return s32[w];
  } else {
    return __funnelshift_r(s32[w], s32[w + 1], 16);
  }
}

// ---- host side -------------------------------------------------------------------------------

// One gather call, as the entry points of roi.cu receive it.
struct GatherArgs {
  const void* image;
  int64_t pitch;              // row pitch in elements; <= 0: W
  int64_t C, T, H, W;
  int itemsize;
  const int32_t* boxes;       // (M,T,2) in elements; null with marker_stride: every box at (0, 0)
  const int32_t* order;       // (M) processing order of the markers, or null
  int64_t marker_stride;      // elements between markers' images (0: all markers share `image`)
  const int32_t* mask_t;      // (T) mask timestep of every timepoint
  int64_t Tm;
  const uint8_t* fg;          // (M,Tm,L,L)
  const uint8_t* bg;
  int64_t M;
  int L;
  void* roi;                  // (M,C,T,L,L); null: summaries only
  bool with_stats;            // summaries into `stats`, or through `peers` when n_peers > 0
  double* stats;              // (M,C,T,kStatsRec)
  const uint64_t* peers;      // host array of n_peers device addresses of (M,C,T,kStatsRec) blocks
  int n_peers;
  int want_median;
  int nf_max = -1, nb_max = -1;   // bounds of the set pixels in any fg / bg mask, -1: unknown

  int64_t row_pitch() const { return pitch > 0 ? pitch : W; }
};

int roi_gather_tma(const GatherArgs& a, cudaStream_t st);     // roi_tma.cu
int roi_gather_lists(const GatherArgs& a, cudaStream_t st);   // roi_lists.cu

extern int g_gather_loader;   // 0 = TMA tensor copies (default), 1 = cp.async chunks
extern int g_gather_wpm;      // warp-per-marker kernels for many-marker shapes

inline PFN_cuTensorMapEncodeTiled get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled>(ptr);
  }
  return fn;
}

// What both staged launchers set up the same way: the window of L rows of wu = L * unit 16-bit units,
// staged wpu = roundup8(wu + 7) units wide (any shift 0..7 plus the row, in whole vectors), the
// tensor map that loads it, and the device limits the launch policies are sized from.
struct StagedWindow {
  TmaGatherParams p;          // the call's pointers and shape, the window geometry and the peer table
  CUtensorMap tmap;
  int max_smem, sm_smem, sms; // shared memory per block (opt-in) and per SM, SM count
};

// MGB_EALIGN when the staged kernels do not apply (the caller falls back), else MGB_OK or an error.
inline int stage_window(const GatherArgs& a, StagedWindow& w) {
  const int unit = a.itemsize / 2;
  const int64_t pitch = a.row_pitch() * unit;   // row pitch in 16-bit units
  const int wu = a.L * unit;
  const int wpu = (wu + 7 + 7) & ~7;
  if ((pitch * 2) % 16 != 0 || !aligned16(a.image) || wpu > 256 || a.L > 256) return MGB_EALIGN;
  if (a.C * a.T > INT32_MAX || a.H > INT32_MAX || pitch > INT32_MAX || a.M > INT32_MAX) return MGB_EALIGN;
  if (a.with_stats && a.Tm > 65535) return MGB_EALIGN;
  PFN_cuTensorMapEncodeTiled encode = get_encode_fn();
  if (!encode) return MGB_EALIGN;
  if (a.n_peers > 8) return MGB_EINVAL;

  TmaGatherParams& p = w.p;
  p = TmaGatherParams{};
  p.roi = (uint16_t*)a.roi; p.boxes = a.boxes; p.order = a.order; p.mask_t = a.mask_t; p.fg = a.fg; p.bg = a.bg;
  p.stats = a.stats;
  p.n_peers = a.n_peers;
  for (int j = 0; j < a.n_peers; ++j) p.peer_stats[j] = reinterpret_cast<double*>(a.peers[j]);
  p.C = a.C; p.T = a.T; p.Tm = a.with_stats ? a.Tm : 1; p.rows = a.L; p.wu = wu; p.wpu = wpu; p.unit = unit;
  p.image = (const uint16_t*)a.image;
  p.H = a.H;
  p.Wu = pitch;
  p.stage_bytes = (a.L * wpu * 2 + 127) & ~127;

  // the tensor covers the whole pitch: the padding columns are real memory, never needed by a window
  const cuuint64_t gdim[3] = {(cuuint64_t)pitch, (cuuint64_t)a.H, (cuuint64_t)(a.C * a.T)};
  const cuuint64_t gstride[2] = {(cuuint64_t)pitch * 2, (cuuint64_t)a.H * pitch * 2};
  const cuuint32_t box[3] = {(cuuint32_t)wpu, (cuuint32_t)a.L, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUresult cr = encode(&w.tmap, CU_TENSOR_MAP_DATA_TYPE_UINT16, 3, const_cast<void*>(a.image), gdim, gstride,
                             box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                             CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) return MGB_EALIGN;

  int dev = 0;
  MGB_CUDA_TRY(cudaGetDevice(&dev));
  MGB_CUDA_TRY(cudaDeviceGetAttribute(&w.max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  MGB_CUDA_TRY(cudaDeviceGetAttribute(&w.sm_smem, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev));
  MGB_CUDA_TRY(cudaDeviceGetAttribute(&w.sms, cudaDevAttrMultiProcessorCount, dev));
  return MGB_OK;
}

// The loop that copies a staged window's rows to the crop.  Rows of one vector or one word would
// divide by 1 (no magic_u32): they take the quads or the word loop, and the element loop.
enum class CopyLoop { kVector, kQuad, kWord, kElement };

// Rows of wu 16-bit units that the word loops copy: an even number of units, more than one word.
inline bool word_rows(int64_t wu) { return wu % 2 == 0 && wu > 2; }

// quads: the caller has an 8-byte quad loop (at most 24 quads per lane) for rows that are not whole vectors
inline CopyLoop copy_loop(int L, int wu, const void* roi, bool quads) {
  const uintptr_t r = reinterpret_cast<uintptr_t>(roi);   // null: summaries only, any loop
  if (wu % 8 == 0 && wu > 8 && (r & 15u) == 0) return CopyLoop::kVector;
  if (quads && wu % 2 == 0 && (L * wu) % 4 == 0 && (r & 7u) == 0 && (L * wu / 4 + 31) / 32 <= 24) return CopyLoop::kQuad;
  if (word_rows(wu) && (r & 3u) == 0) return CopyLoop::kWord;
  return CopyLoop::kElement;
}

// copy_loop for the window of p, with the divisor and magic number of the vector or word loop set in p
inline CopyLoop choose_copy_loop(TmaGatherParams& p, const void* roi, bool quads) {
  const CopyLoop loop = copy_loop(p.rows, p.wu, roi, quads);
  if (loop == CopyLoop::kVector) {
    p.vpr = (uint32_t)(p.wu / 8);
    p.magic_vpr = magic_u32(p.vpr);
  } else if (loop == CopyLoop::kWord) {
    p.half = (uint32_t)(p.wu / 2);
    p.magic_half = magic_u32(p.half);
  }
  return loop;
}

// Host-side record of the last gather launch, read back by mgb_last_gather_path (a diagnostic:
// the launchers write it next to each launch, no kernel reads it).
enum GatherKernel { kGatherListsCta = 1, kGatherListsWpm, kGatherStagedCta, kGatherStagedWpm,
                    kGatherPlainWords, kGatherPlainScalar };
void record_gather_path(GatherKernel kernel, int unroll, CopyLoop loop, int warps, int stages, int loader,
                        bool stats, bool store);   // roi.cu

}  // namespace mgb
