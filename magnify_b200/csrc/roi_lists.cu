// F4 + R with the medians: ROI gather fused with ALL the per-marker reductions the reference's
// consumers run (identify.py:76-80 `where(fg).mean - where(bg).median`, filter.py:21-22,74,82
// medians, filter.py:51 / README.md:21-22 sums and means) in ONE pass over the image.
//
// The windows are staged through shared memory by TMA exactly as in roi_tma.cu.  What differs is
// how the masks are used.  A marker's fg/bg masks are the same for all its (channel, time)
// windows, so they are compacted ONCE per marker into two lists of window offsets (16-bit,
// shared memory).  For every window the warp that owns it
//
//   1. re-aligns and stores the crop (no mask work in that loop),
//   2. loads its share of the masked pixels through the lists into registers, two 16-bit values
//      per register (<= 32 fg + 80 bg values per lane, i.e. fg <= 1024 and bg <= 2560 pixels per
//      marker), and refills its stage with the next window right away,
//   3. sums them (exact integers) and
//   4. finds both exact medians by radix selection on a per-warp shared-memory histogram
//      (warp_median_radix): no block-level synchronisation and no second pass over the crops.
//
// Two work layouts share the code: one CTA per marker with the windows dealt to its warps
// (many windows per marker: chip time series), or one WARP per marker (many markers with few
// windows each: bead screens, time-sharded runs).  Markers whose masks exceed the list
// capacity take the dp2a kernels of roi_tma.cu plus the stand-alone median kernel (roi.cu).
#include <algorithm>

#include "roi_stage.cuh"

namespace mgb {

constexpr int kNFL = 32;   // fg values per lane (16 registers)
constexpr int kNBL = 80;   // bg values per lane (40 registers)

// One (L x L) byte mask, global -> shared memory, with asynchronous copies (all in flight at once;
// the compaction below then reads shared memory instead of paying a DRAM round trip per 32 bytes:
// with one warp per marker that loop was 63 us of the 183 us a config-5 marker took at T = 4).
// Called by `nth` threads (`tid` among them); the caller waits (cp_async_wait_all + barrier).
__device__ __forceinline__ void stage_mask(const uint8_t* __restrict__ g, int n, uint8_t* s, int tid, int nth) {
  const uint32_t sa = smem_u32(s);
  if ((reinterpret_cast<uintptr_t>(g) & 15u) == 0) {
    const int nv = n >> 4;
    for (int i = tid; i < nv; i += nth)
      asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(sa + 16u * i), "l"(g + 16 * i) : "memory");
    for (int i = (nv << 4) + tid; i < n; i += nth) s[i] = g[i];
  } else if ((reinterpret_cast<uintptr_t>(g) & 3u) == 0) {
    const int nv = n >> 2;
    for (int i = tid; i < nv; i += nth)
      asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(sa + 4u * i), "l"(g + 4 * i) : "memory");
    for (int i = (nv << 2) + tid; i < n; i += nth) s[i] = g[i];
  } else {
    for (int i = tid; i < n; i += nth) s[i] = g[i];
  }
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
// generic-proxy accesses to shared memory before this, async-proxy (TMA) writes to it after
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Where the i-th masked pixel (in raster order) sits in the list: within every run of 64, pixel
// 32 h + l goes to position 2 l + h.  A lane's 4-byte load of positions 2 l, 2 l + 1 then brings the
// offsets of pixels l and 32 + l, so each of the two pixel loads that follow reads 32 CONSECUTIVE
// masked pixels across the warp (one row segment, conflict-free) instead of every second one of 64
// (two rows, which collide when the staged row pitch is a multiple of 128 bytes).
__device__ __forceinline__ uint32_t list_slot(uint32_t i) {
  return (i & ~63u) | ((i & 31u) << 1) | ((i >> 5) & 1u);
}

// Compact the non-zero bytes of one (L x L) mask into window offsets row * wpu + col.
// Called by `nwarps` warps (`wi` = this warp's index among them); `cnt` is a shared counter the
// warps advance with one atomic per 32 bytes (nwarps == 1: the count stays in a register).
__device__ __forceinline__ uint32_t build_list(const uint8_t* __restrict__ mask, int L, int wpu, uint32_t magic_l,
                                               uint16_t* list, int cap, int lane, int wi, int nwarps,
                                               uint32_t* cnt) {
  const int total = L * L;
  uint32_t mine = 0;
  for (int base = wi * 32; base < total; base += nwarps * 32) {
    const int e = base + lane;
    const bool on = e < total && mask[e] != 0;
    const unsigned bal = __ballot_sync(0xffffffffu, on);
    if (bal == 0) continue;
    uint32_t start;
    if (nwarps == 1) {
      start = mine;
    } else {
      start = 0;
      if (lane == 0) start = atomicAdd(cnt, (uint32_t)__popc(bal));
      start = __shfl_sync(0xffffffffu, start, 0);
    }
    if (on) {
      const uint32_t pos = start + __popc(bal & ((1u << lane) - 1u));
      const uint32_t row = __umulhi((uint32_t)e, magic_l);
      if (pos < (uint32_t)cap) list[list_slot(pos)] = (uint16_t)(row * wpu + (e - row * L));
    }
    mine += __popc(bal);
  }
  return mine;
}

// Entries [n, cap) repeat entry 0 (offset 0 for an empty mask): every slot of the list is then a
// valid pixel of the window and the per-window loops need no predicates.  The `cap - n` extra
// copies of that pixel are taken out again arithmetically (sum) or from its histogram bin (median).
__device__ __forceinline__ void pad_list(uint16_t* list, uint32_t n, int cap, int tid, int nthreads) {
  const uint16_t fill = n ? list[0] : (uint16_t)0;
  for (int i = (int)n + tid; i < cap; i += nthreads) list[list_slot((uint32_t)i)] = fill;
}

// Bins of the two middle ranks r1 <= r2 in a 256-bin histogram, by a warp scan: lane l owns bins
// 8l .. 8l+7.  before1 = number of values in the bins below bin1.
__device__ __forceinline__ void hist_locate(const uint32_t* hist, int lane, uint32_t r1, uint32_t r2, uint32_t* bin1,
                                            uint32_t* before1, uint32_t* bin2) {
  const uint4 a = reinterpret_cast<const uint4*>(hist)[2 * lane];
  const uint4 b = reinterpret_cast<const uint4*>(hist)[2 * lane + 1];
  const uint32_t c[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  const uint32_t mine = c[0] + c[1] + c[2] + c[3] + c[4] + c[5] + c[6] + c[7];
  uint32_t incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t up = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += up;
  }
  // my candidate answers, valid if the rank falls into my 8 bins
  uint32_t b1 = 0, bf1 = 0, b2 = 0, run = incl - mine;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (r1 >= run && r1 < run + c[j]) { b1 = 8 * lane + j; bf1 = run; }
    if (r2 >= run && r2 < run + c[j]) { b2 = 8 * lane + j; }
    run += c[j];
  }
  const int o1 = __ffs(__ballot_sync(0xffffffffu, incl > r1)) - 1;
  const int o2 = __ffs(__ballot_sync(0xffffffffu, incl > r2)) - 1;
  *bin1 = __shfl_sync(0xffffffffu, b1, o1);
  *before1 = __shfl_sync(0xffffffffu, bf1, o1);
  *bin2 = __shfl_sync(0xffffffffu, b2, o2);
}

// Exact median of the n values a warp holds in v[]: two 16-bit values per register, G groups of
// 4 registers (8 slots) per lane; the slots beyond n hold `pad` extra copies of the value v0.
// Radix selection on a per-warp shared-memory histogram of 256 bins: the values are binned by
// (v - min) >> s with s chosen so that the maximum lands in the last bins, and a warp scan of the
// bin counts locates the bins of the two middle ranks.  With a range below 256 the bins are
// single values and one pass is the answer (typical background: a few dozen grey levels);
// otherwise the bin of the lower middle is binned again at full resolution (2^s <= 256 values),
// or -- when the two middles fall into different bins -- they are the largest value of the one
// and the smallest of the other.  Mean of the two middles for an even count, NaN for n == 0
// (np.nanmedian).
template <int N>
__device__ __forceinline__ double warp_median_radix(const uint32_t (&v)[N], int G, uint32_t n, uint32_t pad,
                                                    uint32_t v0, uint32_t* hist, int lane, uint32_t spill) {
  if (n == 0) return nan_f64();
  uint32_t lo2 = v[0], hi2 = v[0];
#pragma unroll
  for (int g = 0; g < N / 4; ++g) {
    if (g >= G) break;
#pragma unroll
    for (int k = 0; k < 4; ++k) { lo2 = __vminu2(lo2, v[4 * g + k]); hi2 = __vmaxu2(hi2, v[4 * g + k]); }
  }
  uint32_t lo = min(lo2 & 0xffffu, lo2 >> 16), hi = max(hi2 & 0xffffu, hi2 >> 16);
  lo = __reduce_min_sync(0xffffffffu, lo);
  hi = __reduce_max_sync(0xffffffffu, hi);
  if (lo == hi) return (double)lo;
  const uint32_t r1 = (n - 1u) >> 1, r2 = n >> 1;  // ranks of the lower / upper middle (equal for odd n)
  const int bits = 32 - __clz(hi - lo);
  const int s = bits > 8 ? bits - 8 : 0;
  uint4* h4 = reinterpret_cast<uint4*>(hist);
  h4[2 * lane] = make_uint4(0, 0, 0, 0);
  h4[2 * lane + 1] = make_uint4(0, 0, 0, 0);
  __syncwarp();
#pragma unroll
  for (int g = 0; g < N / 4; ++g) {
    if (g >= G) break;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t w = v[4 * g + k];
      atomicAdd(hist + (((w & 0xffffu) - lo) >> s), 1u);
      atomicAdd(hist + (((w >> 16) - lo) >> s), 1u);
    }
  }
  __syncwarp();
  if (lane == 0 && pad) hist[(v0 - lo) >> s] -= pad;
  __syncwarp();
  uint32_t bin1, before1, bin2;
  hist_locate(hist, lane, r1, r2, &bin1, &before1, &bin2);
  if (s == 0) return 0.5 * ((double)(lo + bin1) + (double)(lo + bin2));
  if (bin1 != bin2) {
    uint32_t a = 0, b = 0xffffffffu;
#pragma unroll
    for (int g = 0; g < N / 4; ++g) {
      if (g >= G) break;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t w = v[4 * g + k];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const uint32_t x = h ? (w >> 16) : (w & 0xffffu), bin = (x - lo) >> s;
          a = max(a, bin == bin1 ? x : 0u);
          b = min(b, bin == bin2 ? x : 0xffffffffu);
        }
      }
    }
    a = __reduce_max_sync(0xffffffffu, a);
    b = __reduce_min_sync(0xffffffffu, b);
    return 0.5 * ((double)a + (double)b);
  }
  // both middles in one coarse bin: bin its 2^s values exactly (everything else goes to the lane's own
  // slot behind the 256 bins that are read back)
  const uint32_t base = lo + (bin1 << s), width = 1u << s;
  __syncwarp();
  h4[2 * lane] = make_uint4(0, 0, 0, 0);
  h4[2 * lane + 1] = make_uint4(0, 0, 0, 0);
  __syncwarp();
#pragma unroll
  for (int g = 0; g < N / 4; ++g) {
    if (g >= G) break;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t w = v[4 * g + k];
      const uint32_t d0 = (w & 0xffffu) - base, d1 = (w >> 16) - base;
      atomicAdd(hist + (d0 < 256u ? d0 : spill), 1u);      // slots 256.. = "not in this bin", one per lane (no conflicts)
      atomicAdd(hist + (d1 < 256u ? d1 : spill), 1u);
    }
  }
  __syncwarp();
  if (lane == 0 && pad && v0 - base < width) hist[v0 - base] -= pad;
  __syncwarp();
  uint32_t f1, unused, f2;
  hist_locate(hist, lane, r1 - before1, r2 - before1, &f1, &unused, &f2);
  return 0.5 * ((double)(base + f1) + (double)(base + f2));
}

constexpr int kHistWords = 256 + 32;   // 256 bins + one overflow slot per lane

// VPL > 0: rows are whole 16-byte vectors, the copy loop is unrolled (VPL vectors per lane).
// QPL > 0: rows of an even number of pixels copied as 8-byte quads (QPL quads per lane).
// both 0 : run-time loops (vector rows of any size, word rows, odd rows).
// WPM    : one warp per marker instead of one CTA per marker.   NW: warps per CTA (launch bound).
template <int VPL, int QPL, bool WPM, int NW>
__global__ void __launch_bounds__(NW * 32, NW == 6 ? 2 : 1)
roi_gather_lists_kernel(const __grid_constant__ CUtensorMap tmap, const TmaGatherParams p, int64_t M,
                        uint32_t magic_l) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nw = blockDim.x >> 5;
  const int tm = blockIdx.y;
  const int groups = WPM ? nw : 1;            // markers per CTA
  const int g = WPM ? warp : 0;

  uint8_t* stages = smem;                                                   // [warp][stage][stage_bytes]
  uint16_t* lists = reinterpret_cast<uint16_t*>(stages + (size_t)nw * p.n_stages * p.stage_bytes);
  uint32_t* hists = reinterpret_cast<uint32_t*>(lists + (size_t)groups * (p.cap_f + p.cap_b));  // [warp][kHistWords]
  uint64_t* bars = reinterpret_cast<uint64_t*>(hists + (size_t)nw * kHistWords);                // [warp][4]
  int32_t* tlist = reinterpret_cast<int32_t*>(bars + (size_t)nw * 4);       // timepoints of this mask timestep
  __shared__ int s_nt;
  __shared__ uint32_t s_cnt[2];

  if (warp == 0) {
    int n = 0;
    for (int64_t base = 0; base < p.T; base += 32) {
      const int64_t t = base + lane;
      const bool hit = (t < p.T) && p.mask_t[t] == tm;
      const unsigned bal = __ballot_sync(0xffffffffu, hit);
      if (hit) tlist[n + __popc(bal & ((1u << lane) - 1))] = (int32_t)t;
      n += __popc(bal);
    }
    if (lane == 0) { s_nt = n; s_cnt[0] = 0; s_cnt[1] = 0; }
  }
  if (lane == 0) {
    for (int s = 0; s < p.n_stages; ++s) mbar_init(smem_u32(&bars[warp * 4 + s]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  // CTA layout: CTA b < split_from works on all the windows of marker b; the markers from
  // split_from on (the ones that would run as a nearly empty last wave) are shared by split_parts
  // CTAs each, which deal the marker's rounds of nw windows among themselves.
  int64_t mi = WPM ? (int64_t)blockIdx.x * nw + warp : (int64_t)blockIdx.x;
  int part = 0, nparts = 1;
  if (!WPM && mi >= p.split_from) {
    const int64_t r = mi - p.split_from;
    mi = p.split_from + r / p.split_parts;
    part = (int)(r % p.split_parts);
    nparts = p.split_parts;
  }
  const bool active = mi < M;
  const int64_t m = active ? (p.order ? p.order[mi] : mi) : 0;
  uint16_t* fl = lists + (size_t)g * (p.cap_f + p.cap_b);
  uint16_t* bl = fl + p.cap_f;
  uint32_t nf = 0, nb = 0;
  // the two masks go through the (still unused) window stages: the warp's own in the warp layout,
  // the start of the stage area in the CTA layout (a stage holds rows x wpu x 2 >= 2 x rows^2 bytes)
  const int mask_len = p.rows * p.rows, mask_room = (mask_len + 15) & ~15;
  uint8_t* mstage = stages + (WPM ? (size_t)warp * p.n_stages * p.stage_bytes : 0);
  if (active) {
    const uint8_t* f = p.fg + (m * p.Tm + tm) * (int64_t)mask_len;
    const uint8_t* b = p.bg + (m * p.Tm + tm) * (int64_t)mask_len;
    stage_mask(f, mask_len, mstage, WPM ? lane : (int)threadIdx.x, WPM ? 32 : (int)blockDim.x);
    stage_mask(b, mask_len, mstage + mask_room, WPM ? lane : (int)threadIdx.x, WPM ? 32 : (int)blockDim.x);
  }
  cp_async_wait_all();
  __syncthreads();
  if (active) {
    nf = build_list(mstage, p.rows, p.wpu, magic_l, fl, p.cap_f, lane, WPM ? 0 : warp, WPM ? 1 : nw, &s_cnt[0]);
    nb = build_list(mstage + mask_room, p.rows, p.wpu, magic_l, bl, p.cap_b, lane, WPM ? 0 : warp, WPM ? 1 : nw,
                    &s_cnt[1]);
  }
  fence_proxy_async_smem();
  __syncthreads();
  if (!WPM) { nf = s_cnt[0]; nb = s_cnt[1]; }
  // a mask larger than the lists cannot happen when the caller sized them from the masks
  // (mgb_mask_count_max); if it does, the sums / medians of this marker are flagged NaN
  const bool overflow = nf > (uint32_t)p.cap_f || nb > (uint32_t)p.cap_b;
  if (active && !overflow) {
    pad_list(fl, nf, p.cap_f, WPM ? lane : (int)threadIdx.x, WPM ? 32 : (int)blockDim.x);
    pad_list(bl, nb, p.cap_b, WPM ? lane : (int)threadIdx.x, WPM ? 32 : (int)blockDim.x);
  }
  __syncthreads();
  if (!active) return;
  const double cnt_fg = (double)nf, cnt_bg = (double)nb;
  const int GF = p.cap_f >> 8, GB = p.cap_b >> 8;       // groups of 8 slots per lane (256 values); uniform
  const uint32_t pad_f = (uint32_t)p.cap_f - nf, pad_b = (uint32_t)p.cap_b - nb;

  const int nt = s_nt;
  const int n_items = nt * (int)p.C;           // item i -> (c = i / nt, t = tlist[i % nt])

  // The per-lane shared-memory offsets of the copy loop do not depend on the window, but keeping
  // them in registers across the medians (21 to 48 of them) costs more than recomputing them per
  // window with a multiply-high; `opaque` keeps the compiler from hoisting them out of the loop.
  constexpr int kV = VPL > 0 ? VPL : 1;
  const int nquads = (p.rows * p.wu) >> 2;

  uint8_t* my_stages = stages + (size_t)warp * p.n_stages * p.stage_bytes;
  const uint32_t my_stage0 = smem_u32(my_stages);
  const uint32_t my_bar0 = smem_u32(&bars[warp * 4]);
  uint32_t* my_hist = hists + (size_t)warp * kHistWords;
  const uint32_t tx_bytes = (uint32_t)(p.rows * p.wpu * 2);
  const int first = WPM ? 0 : part * nw + warp, step = WPM ? 1 : nparts * nw;

  // (channel, index into tlist) of an item, advanced without divisions
  struct Cursor { int i, c, k; };
  auto advance = [&](Cursor& cur, int by) {
    cur.i += by;
    cur.k += by;
    while (cur.k >= nt) { cur.k -= nt; ++cur.c; }
  };
  auto issue_tma = [&](const Cursor& cur, int s) {
    if (lane == 0) {
      const int64_t t = tlist[cur.k];
      const int32_t top = p.boxes[(m * p.T + t) * 2];
      const int32_t left = p.boxes[(m * p.T + t) * 2 + 1];
      const uint32_t bar = my_bar0 + s * 8;
      mbar_expect_tx(bar, tx_bytes);
      tma_load_3d(my_stage0 + s * p.stage_bytes, &tmap, bar, left & ~7, top, (int)(cur.c * p.T + t));
    }
  };

  Cursor ahead{0, 0, 0}, cur{0, 0, 0};
  if (nt > 0) { advance(ahead, first); advance(cur, first); }
  // every stage holds a window in flight; a stage is refilled as soon as its window has been copied
  // out and its masked pixels sit in registers, i.e. BEFORE the medians of that window are worked
  // out -- so even a single stage per warp overlaps its next load with half of the work
  for (int s = 0; s < p.n_stages; ++s) {
    if (ahead.i < n_items) issue_tma(ahead, s);
    if (nt > 0) advance(ahead, step);
  }
  int s = 0;
  uint32_t parity = 0;
  for (; cur.i < n_items; advance(cur, step)) {
    const int64_t c = cur.c, t = tlist[cur.k];
    const int shift = p.boxes[(m * p.T + t) * 2 + 1] & 7;
    const int64_t n = (m * p.C + c) * p.T + t;
    const uint8_t* buf = my_stages + (size_t)s * p.stage_bytes;
    mbar_wait(my_bar0 + s * 8, parity);

    // ---- 1. the crop
    if (p.store) {
      uint16_t* dst = p.roi + n * (int64_t)p.rows * p.wu;
      uint32_t opaque = 0;
      asm volatile("" : "+r"(opaque));
      if constexpr (QPL > 0) {
        uint2* d2 = reinterpret_cast<uint2*>(dst);
        const uint32_t* s32 = reinterpret_cast<const uint32_t*>(buf);
        auto copy = [&](auto par) {
          constexpr int PAR = decltype(par)::value;
#pragma unroll
          for (int k = 0; k < QPL; ++k) {
            const int q = lane + 32 * k;
            if (q < nquads) {
              const uint32_t u = 4u * q + opaque;
              const uint32_t row = __umulhi(u, p.magic_wu), col = u - row * p.wu;
              const uint32_t oa = row * p.wpu + col + shift;
              const uint32_t ob = (col + 2 < (uint32_t)p.wu) ? oa + 2 : (row + 1) * p.wpu + shift;   // second pair wraps to the next row
              const uint32_t lo = load_pair<PAR>(s32, oa);
              const uint32_t hi = load_pair<PAR>(s32, ob);
              asm volatile("st.global.L1::no_allocate.v2.u32 [%0], {%1,%2};" ::"l"(d2 + q), "r"(lo), "r"(hi) : "memory");
            }
          }
        };
        if (shift & 1) copy(std::integral_constant<int, 1>{});
        else copy(std::integral_constant<int, 0>{});
      } else {
        uint32_t dummy_f, dummy_b;
        if (p.vpr) {
          uint32_t svo[kV];
          if constexpr (VPL > 0) {
            const uint32_t nvec = p.rows * p.vpr, pitch = p.wpu >> 3;
#pragma unroll
            for (int k = 0; k < VPL; ++k) {
              const uint32_t v = lane + 32 * k;
              const uint32_t vv = (v < nvec ? v : 0) + opaque;
              const uint32_t row = __umulhi(vv, p.magic_vpr);
              svo[k] = row * pitch + (vv - row * p.vpr);
            }
          }
          switch (shift) {
#define MGB_COPY(SS) \
  case SS: consume_vec<false, true, SS, VPL>(p, buf, dst, nullptr, nullptr, lane, nullptr, nullptr, svo, &dummy_f, &dummy_b); break;
            MGB_COPY(0) MGB_COPY(1) MGB_COPY(2) MGB_COPY(3) MGB_COPY(4) MGB_COPY(5) MGB_COPY(6)
            default: consume_vec<false, true, 7, VPL>(p, buf, dst, nullptr, nullptr, lane, nullptr, nullptr, svo, &dummy_f, &dummy_b); break;
#undef MGB_COPY
          }
        } else {
          consume_generic<false, true>(p, buf, dst, nullptr, nullptr, lane, shift, &dummy_f, &dummy_b);
        }
      }
    }

    double dsf = nan_f64(), dsb = nan_f64(), mf = nan_f64(), mb = nan_f64();
    if (overflow) {
      __syncwarp();
      if (ahead.i < n_items) issue_tma(ahead, s);
      advance(ahead, step);
    } else {
      // ---- 2. + 3. the masked pixels of this window through the lists (every slot is a valid
      // pixel: the slots beyond the mask repeat the mask's first pixel)
      const uint16_t* s16 = reinterpret_cast<const uint16_t*>(buf) + shift;
      // slots 2q, 2q+1 of group g read list positions 256 g + 64 q + 2 lane (+1): one 4-byte load brings
      // two offsets per lane (a full 128-byte wavefront for the warp); by list_slot() they are masked
      // pixels 64 q' + lane and 64 q' + 32 + lane, so each pixel load covers 32 consecutive masked pixels
      const uint32_t* flg = reinterpret_cast<const uint32_t*>(fl) + lane;
      const uint32_t* blg = reinterpret_cast<const uint32_t*>(bl) + lane;
      uint32_t vf[kNFL / 2], vb[kNBL / 2];                  // two 16-bit values per register
      uint32_t sf = 0, sb = 0;
#pragma unroll
      for (int gi = 0; gi < kNFL / 8; ++gi) {
        if (gi >= GF) break;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint32_t o2 = flg[128 * gi + 32 * q];
          const uint32_t w = (uint32_t)s16[o2 & 0xffffu] | ((uint32_t)s16[o2 >> 16] << 16);
          vf[4 * gi + q] = w;
          sf = __dp2a_lo(w, 0x0101u, sf);                    // both halves added (exact: <= 112 x 65535 per lane)
        }
      }
#pragma unroll
      for (int gi = 0; gi < kNBL / 8; ++gi) {
        if (gi >= GB) break;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint32_t o2 = blg[128 * gi + 32 * q];
          const uint32_t w = (uint32_t)s16[o2 & 0xffffu] | ((uint32_t)s16[o2 >> 16] << 16);
          vb[4 * gi + q] = w;
          sb = __dp2a_lo(w, 0x0101u, sb);
        }
      }
      const uint32_t v0f = s16[fl[0]], v0b = s16[bl[0]];     // the pixel the padding repeats
      __syncwarp();                                          // every lane is done with the staged window
      if (ahead.i < n_items) issue_tma(ahead, s);
      advance(ahead, step);
      sf = __reduce_add_sync(0xffffffffu, sf) - pad_f * v0f;
      sb = __reduce_add_sync(0xffffffffu, sb) - pad_b * v0b;
      dsf = (double)sf;
      dsb = (double)sb;
      // ---- 4. medians
      if (p.want_median) {
        const uint32_t spill = 256u + (uint32_t)lane;   // this lane's slot for "not in the bin" (no conflicts)
        mf = warp_median_radix(vf, GF, nf, pad_f, v0f, my_hist, lane, spill);
        __syncwarp();
        mb = warp_median_radix(vb, GB, nb, pad_b, v0b, my_hist, lane, spill);
      }
    }
    write_stats(p, lane, n, cnt_fg, cnt_bg, dsf, dsb, mf, mb);
    __syncwarp();
    if (++s == p.n_stages) { s = 0; parity ^= 1; }
  }
}

// Largest number of non-zero bytes in any fg mask and in any bg mask: what the list capacities of
// the kernel above are sized from.  One warp per (marker, mask timestep).
__global__ void __launch_bounds__(kThreads)
mask_count_max_kernel(const uint8_t* __restrict__ fg, const uint8_t* __restrict__ bg, int64_t n_masks, int64_t len,
                      int32_t* __restrict__ out) {
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= n_masks) return;
  const uint8_t* f = fg + w * len;
  const uint8_t* b = bg + w * len;
  uint32_t cf = 0, cb = 0;
  for (int64_t i = lane; i < len; i += 32) {
    cf += f[i] != 0;
    cb += b[i] != 0;
  }
  cf = __reduce_add_sync(0xffffffffu, cf);
  cb = __reduce_add_sync(0xffffffffu, cb);
  if (lane == 0) {
    atomicMax(out, (int32_t)cf);
    atomicMax(out + 1, (int32_t)cb);
  }
}

PFN_cuTensorMapEncodeTiled get_encode_fn();   // roi_tma.cu
extern int g_gather_wpm;

static uint32_t magic_u32_(uint32_t d) { return (uint32_t)((0x100000000ULL + d - 1) / d); }

// Returns MGB_OK when launched, MGB_EALIGN when this path does not apply (the caller falls back
// to the dp2a kernels, which leave the median columns NaN), or an error.
int roi_gather_lists(const void* image, int64_t pitch, int64_t C, int64_t T, int64_t H, int64_t W,
                     const int32_t* boxes, const int32_t* order, const int32_t* mask_t, int64_t Tm, const uint8_t* fg,
                     const uint8_t* bg, int64_t M, int L, void* roi, double* stats, int want_median, int nf_max,
                     int nb_max, const uint64_t* host_peers, int n_peers, cudaStream_t st) {
  if (!stats || nf_max < 0 || nb_max < 0) return MGB_EALIGN;
  if (nf_max > kNFL * 32 || nb_max > kNBL * 32) return MGB_EALIGN;
  const int wu = L;
  const int wpu = (wu + 7 + 7) & ~7;
  if ((pitch * 2) % 16 != 0 || !aligned16(image) || wpu > 256 || L > 256) return MGB_EALIGN;
  if ((int64_t)(L - 1) * wpu + L + 8 > 65535) return MGB_EALIGN;      // list entries are 16-bit offsets
  if (C * T > INT32_MAX || H > INT32_MAX || pitch > INT32_MAX || M > INT32_MAX || Tm > 65535) return MGB_EALIGN;
  PFN_cuTensorMapEncodeTiled encode = get_encode_fn();
  if (!encode) return MGB_EALIGN;

  TmaGatherParams p{};
  p.roi = (uint16_t*)roi; p.boxes = boxes; p.order = order; p.mask_t = mask_t; p.fg = fg; p.bg = bg; p.stats = stats;
  p.C = C; p.T = T; p.Tm = Tm; p.rows = L; p.wu = wu; p.wpu = wpu; p.unit = 1;
  p.n_peers = 0;
  if (host_peers && n_peers > 0) {
    if (n_peers > 8) return MGB_EINVAL;
    p.n_peers = n_peers;
    for (int j = 0; j < n_peers; ++j) p.peer_stats[j] = reinterpret_cast<double*>(host_peers[j]);
  }
  p.stage_bytes = (L * wpu * 2 + 127) & ~127;
  p.cap_f = (std::max(nf_max, 1) + 255) & ~255;     // whole groups of 8 slots per lane
  p.cap_b = (std::max(nb_max, 1) + 255) & ~255;
  p.want_median = want_median ? 1 : 0;
  p.store = roi ? 1 : 0;
  const bool out16 = !roi || aligned16(roi);
  const bool out8 = !roi || (reinterpret_cast<uintptr_t>(roi) & 7u) == 0;
  const bool out4 = !roi || (reinterpret_cast<uintptr_t>(roi) & 3u) == 0;
  int vpl = 0, qpl = 0;
  // the copy loops divide by vpr / half with a multiply-high by ceil(2^32 / d), which has no 32-bit
  // value for d = 1: rows of one vector (L = 8) take the quads, rows of one word (L = 2) the generic loop
  if (wu % 8 == 0 && wu > 8 && out16) {
    p.vpr = (uint32_t)(wu / 8);
    p.magic_vpr = magic_u32_(p.vpr);
    const int v = (int)((L * p.vpr + 31) / 32);
    vpl = v <= 12 ? 12 : v <= 21 ? 21 : v <= 36 ? 36 : 0;
  } else if (wu % 2 == 0 && (L * wu) % 4 == 0 && out8 && (L * wu / 4 + 31) / 32 <= 24) {
    qpl = (L * wu / 4 + 31) / 32 <= 12 ? 12 : 24;
  } else if (wu % 2 == 0 && wu > 2 && out4) {
    p.half = (uint32_t)(wu / 2);
    p.magic_half = magic_u32_(p.half);
  }

  // Work layout: one CTA per marker when every marker has many windows, one warp per marker
  // when it has few and there are enough markers to fill the machine.
  const int64_t items = C * std::max<int64_t>(1, T / std::max<int64_t>(1, Tm));
  int dev = 0, max_smem = 0, sms = 0;
  MGB_CUDA_TRY(cudaGetDevice(&dev));
  MGB_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  MGB_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  // (a warp per marker needs many more markers than warp slots, else the last wave runs half empty:
  // 1792 markers on 148 x 12 slots took 2.25 ms in that layout against 1.15 ms with a CTA per marker.
  // Handing every warp an equal run of the flattened (marker, window) space instead was tried and
  // is slower still -- 3.9 ms against 2.0 ms at config 3, 14.1 against 10.3 ms at config 5 T = 4:
  // 1776 warps then write crops into 1776 regions megabytes apart at once.)
  bool wpm = g_gather_wpm && items < 128 && M * Tm >= (int64_t)sms * 12 * 8;
  if (const char* e = getenv("MGB_GATHER_LAYOUT")) wpm = atoi(e) == 1 ? true : atoi(e) == 0 ? false : wpm;   // tuning only

  const size_t list_bytes = (size_t)(p.cap_f + p.cap_b) * sizeof(uint16_t);
  int sm_smem = 0;
  MGB_CUDA_TRY(cudaDeviceGetAttribute(&sm_smem, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev));
  int nw = 0, ns = 0;
  size_t smem_bytes = 0;
  // warps per CTA x stages per warp: more warps hide the latency of the per-window reductions,
  // more stages that of the window loads; 12 x 1 ... 8 x 2 ... 4 x 2 in order of preference.
  // The warp layout (small windows, dense masks: latency-bound) takes 16 warps at 128 registers when
  // they fit (config 5: 13.2 against 14.9 ms); the CTA layout at config 3 is memory-bound and loses
  // with 16 (1.98 against 1.80 ms: the spills of the 128-register build cost more than the warps gain).
  // With a CTA per marker and fewer than 128 windows per marker, two CTAs of 6 warps share an SM
  // instead: the list building of one overlaps the windows of the other and fewer warps idle in
  // a marker's last round (config 3: 0.46 against 0.54 ms at T = 7, 1.12 against 1.17 ms at
  // T = 25, 2.06 against 2.03 ms at T = 50).
  int want_nw = 0;
  if (const char* e = getenv("MGB_GATHER_WARPS")) want_nw = atoi(e);   // tuning only
  for (int pass = 0; pass < 2 && !nw; ++pass) {
    const bool pair = !wpm && items < 128;
    for (int cand : {6, 16, 12, 8, 4}) {
      if (want_nw ? cand != want_nw : ((cand == 6 && !pair) || (cand == 16 && !wpm))) continue;
      const size_t fixed = (wpm ? cand : 1) * list_bytes + (size_t)cand * kHistWords * sizeof(uint32_t) +
                           (size_t)cand * 4 * sizeof(uint64_t) + (size_t)T * sizeof(int32_t) + 128;
      // 6 warps: two CTAs share an SM (half of its shared memory each, 1 KB reserved per CTA)
      const size_t room = cand == 6 ? (size_t)(sm_smem / 2 - 1024) : (size_t)max_smem;
      if (room < fixed + 1024) continue;
      const bool one = cand >= 12 || cand == 6;
      const int n = (int)std::min<size_t>(one ? 1 : 4, (room - fixed - 1024) / ((size_t)cand * p.stage_bytes));
      if (n >= (one ? 1 : 2)) { nw = cand; ns = n; smem_bytes = (size_t)cand * n * p.stage_bytes + fixed; break; }
    }
    if (!nw && wpm) wpm = false;   // per-warp lists do not fit: share one marker per CTA instead
  }
  if (!nw) return MGB_EALIGN;
  bool split_tail = true;
  if (const char* e = getenv("MGB_GATHER_SPLIT")) split_tail = atoi(e) != 0;   // tuning / tests only
  p.n_stages = ns;
  p.magic_wu = magic_u32_((uint32_t)wu);

  CUtensorMap tmap;
  const cuuint64_t gdim[3] = {(cuuint64_t)pitch, (cuuint64_t)H, (cuuint64_t)(C * T)};
  const cuuint64_t gstride[2] = {(cuuint64_t)pitch * 2, (cuuint64_t)H * pitch * 2};
  const cuuint32_t box[3] = {(cuuint32_t)wpu, (cuuint32_t)L, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUresult cr = encode(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT16, 3, const_cast<void*>(image), gdim, gstride, box,
                             estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                             CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) return MGB_EALIGN;
  p.image = (const uint16_t*)image;
  p.H = H;
  p.Wu = pitch;

  const uint32_t magic_l = magic_u32_((uint32_t)L);
  // CTA layout: with M markers on `slots` resident CTAs the last M % slots markers would run as a
  // wave that leaves most SMs idle for a whole marker's duration (config 3: 1792 = 12 x 148 + 16).
  // Those markers are split over up to 8 CTAs each, so that the last wave is short.
#define MGB_LAUNCH_L(VP, QP, WP, NWARPS)                                                                   \
  do {                                                                                                    \
    auto kern = roi_gather_lists_kernel<VP, QP, WP, NWARPS>;                                              \
    MGB_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes)); \
    dim3 grid(WP ? (unsigned)((M + nw - 1) / nw) : (unsigned)M, (unsigned)Tm);                            \
    p.split_from = M;                                                                                     \
    p.split_parts = 1;                                                                                    \
    if (!WP && split_tail) {                                                                          \
      int resident = 1;                                                                                   \
      MGB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kern, nw * 32, smem_bytes));  \
      const int64_t slots = (int64_t)std::max(resident, 1) * sms, tail = (M * Tm) % slots;                \
      const int64_t rounds = (items + nw - 1) / nw;                                                       \
      const int parts = (int)std::min<int64_t>({8, tail ? slots / tail : 1, rounds});                     \
      if (Tm == 1 && M > slots && parts >= 2) {                                                           \
        p.split_from = M - tail;                                                                          \
        p.split_parts = parts;                                                                            \
        grid.x = (unsigned)(p.split_from + tail * parts);                                                 \
      }                                                                                                   \
    }                                                                                                     \
    kern<<<grid, nw * 32, smem_bytes, st>>>(tmap, p, M, magic_l);                                         \
  } while (0)
#define MGB_LAUNCH_NW(VP, QP, WP)                       \
  do {                                                  \
    if (nw == 16) MGB_LAUNCH_L(VP, QP, WP, 16);         \
    else if (nw == 12) MGB_LAUNCH_L(VP, QP, WP, 12);    \
    else if (nw == 6) MGB_LAUNCH_L(VP, QP, WP, 6);      \
    else MGB_LAUNCH_L(VP, QP, WP, 8);                   \
  } while (0)
#define MGB_LAUNCH_CP(WP)                        \
  do {                                           \
    if (vpl == 12) MGB_LAUNCH_NW(12, 0, WP);     \
    else if (vpl == 21) MGB_LAUNCH_NW(21, 0, WP);\
    else if (vpl == 36) MGB_LAUNCH_NW(36, 0, WP);\
    else if (qpl == 12) MGB_LAUNCH_NW(0, 12, WP);\
    else if (qpl == 24) MGB_LAUNCH_NW(0, 24, WP);\
    else MGB_LAUNCH_NW(0, 0, WP);                \
  } while (0)
  if (wpm) MGB_LAUNCH_CP(true);
  else MGB_LAUNCH_CP(false);
#undef MGB_LAUNCH_NW
#undef MGB_LAUNCH_CP
#undef MGB_LAUNCH_L
  MGB_CUDA_LAUNCH_CHECK();
  return MGB_OK;
}

}  // namespace mgb

using namespace mgb;

extern "C" int mgb_mask_count_max(const uint8_t* fg, const uint8_t* bg, int64_t n_masks, int64_t mask_len,
                                  int32_t* counts, void* stream) {
  if (n_masks < 0 || mask_len < 0 || !counts) return MGB_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  MGB_CUDA_TRY(cudaMemsetAsync(counts, 0, 2 * sizeof(int32_t), st));
  if (n_masks == 0 || mask_len == 0) return MGB_OK;
  if (!fg || !bg) return MGB_EINVAL;
  const int64_t blocks = ceil_div(n_masks * 32, kThreads);
  if (blocks > INT32_MAX) return MGB_EUNSUPPORTED;
  mask_count_max_kernel<<<(unsigned)blocks, kThreads, 0, st>>>(fg, bg, n_masks, mask_len, counts);
  MGB_CUDA_LAUNCH_CHECK();
  return MGB_OK;
}
