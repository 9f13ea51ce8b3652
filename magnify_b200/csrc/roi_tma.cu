// F4 + R, TMA path: ROI windows are staged through shared memory by the tensor-memory
// accelerator (cp.async.bulk.tensor, SASS UTMALDG); the warp that owns a window re-aligns it
// out of shared memory with 128-bit loads + a funnel shift, stores it with aligned 128-bit
// streaming stores and accumulates the masked sums (dp2a) from the same registers.
//
// Measured constraint (tools/tma_probe2.cu on B200): a tiled TMA load faults ("illegal
// instruction") unless coordinate[0] * elemsize is a multiple of 16 bytes.  ROI windows start at
// arbitrary pixels, so the box is widened to start at the 16-byte boundary below `left` and the
// residual shift (0..7 pixels, uniform per window) is applied while reading shared memory.
//
// One CTA = one marker m (x one mask timestep); its warps share the marker's fg/bg masks in
// shared memory and each runs an independent NS-stage pipeline over its (channel, time) items:
//
//     lane 0:  expect_tx + TMA load of item k+NS-1  --->  mbarrier full[s]
//     warp  :  wait full[s] -> realign + store roi[m,c,t] + masked sums
//     lane 0:  (after __syncwarp) refill the stage item k-1 used
//
// Reference semantics: roi[m,c,t] = image[c,t, top:top+L, left:left+L] (find.py:160-169,
// 324-334, 589-602); sums/means over fg/bg (identify.py:76-80, filter.py:21-22,51).
#include "roi_stage.cuh"

namespace mgb {

template <bool STATS, bool STORE, int VPL>
__global__ void __launch_bounds__(kTmaMaxWarps * 32, 1)
roi_gather_tma_kernel(const __grid_constant__ CUtensorMap tmap, const TmaGatherParams p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nw = blockDim.x >> 5;
  // Markers may be visited in a caller-given order (spatially sorted: CTAs that run together then
  // touch neighbouring image rows, and DRAM lines shared by overlapping windows hit in L2).
  const int64_t m = p.order ? p.order[blockIdx.x] : blockIdx.x;
  const int tm = blockIdx.y;

  // shared memory carve-up
  uint8_t* stages = smem;                                                  // [warp][stage][stage_bytes]
  const int mask_bytes = STATS ? ((p.rows * p.wu + 15) & ~15) : 0;         // dense (rows x wu), 1 B / unit
  uint8_t* fgm = stages + (size_t)nw * p.n_stages * p.stage_bytes;
  uint8_t* bgm = fgm + mask_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(bgm + mask_bytes);          // [warp][8]
  int32_t* tlist = reinterpret_cast<int32_t*>(bars + kTmaMaxWarps * 8);    // timepoints of this CTA
  __shared__ int s_nt;
  __shared__ uint32_t s_cnt[2][kTmaMaxWarps];

  if (warp == 0) {
    const int n = list_timepoints<STATS>(p, tm, tlist, lane);
    if (lane == 0) s_nt = n;
  }
  if constexpr (STATS) {
    // masks of (m, tm) expanded to one byte per 16-bit unit; counts are per element
    const uint8_t* f = p.fg + (m * p.Tm + tm) * (int64_t)p.rows * p.rows;
    const uint8_t* b = p.bg + (m * p.Tm + tm) * (int64_t)p.rows * p.rows;
    uint32_t nf = 0, nb = 0;
    const int total = p.rows * p.wu;
    for (int i = threadIdx.x; i < mask_bytes; i += blockDim.x) {
      uint8_t vf = 0, vb = 0;
      if (i < total) {
        const int row = i / p.wu, col = i - row * p.wu;
        const int e = row * p.rows + col / p.unit;
        vf = f[e] != 0;
        vb = b[e] != 0;
        if (col % p.unit == 0) { nf += vf; nb += vb; }
      }
      fgm[i] = vf;
      bgm[i] = vb;
    }
    nf = __reduce_add_sync(0xffffffffu, nf);
    nb = __reduce_add_sync(0xffffffffu, nb);
    if (lane == 0) { s_cnt[0][warp] = nf; s_cnt[1][warp] = nb; }
  }
  if (p.loader == 0 && lane == 0) init_stage_barriers(&bars[warp * 8], p.n_stages);
  __syncthreads();
  const int nt = s_nt;
  const int n_items = nt * (int)p.C;           // item i -> (c = i / nt, t = tlist[i % nt])
  double cnt_fg = 0.0, cnt_bg = 0.0;
  if constexpr (STATS) {
    uint32_t a = 0, c = 0;
    for (int i = 0; i < nw; ++i) { a += s_cnt[0][i]; c += s_cnt[1][i]; }
    cnt_fg = (double)a;
    cnt_bg = (double)c;
  }

  // window-independent per-lane state of the unrolled vector path
  constexpr int kV = VPL > 0 ? VPL : 1;
  uint2 fm[kV], bm[kV];
  uint32_t svo[kV];
  if constexpr (VPL > 0) {
    const uint32_t nvec = p.rows * p.vpr, pitch = p.wpu >> 3;
#pragma unroll
    for (int k = 0; k < VPL; ++k) {
      const uint32_t v = lane + 32 * k;
      const uint32_t vv = v < nvec ? v : 0;
      const uint32_t row = __umulhi(vv, p.magic_vpr);
      svo[k] = row * pitch + (vv - row * p.vpr);
      if constexpr (STATS) {
        fm[k] = reinterpret_cast<const uint2*>(fgm)[vv];
        bm[k] = reinterpret_cast<const uint2*>(bgm)[vv];
      } else {
        fm[k] = make_uint2(0, 0);
        bm[k] = make_uint2(0, 0);
      }
    }
  }

  uint8_t* my_stages = stages + (size_t)warp * p.n_stages * p.stage_bytes;
  const uint32_t my_stage0 = smem_u32(my_stages);
  const uint32_t my_bar0 = smem_u32(&bars[warp * 8]);
  const uint32_t tx_bytes = (uint32_t)(p.rows * p.wpu * 2);
  const int cpr = p.wpu >> 3;                   // 16-byte chunks per staged row
  const int n_chunks = p.rows * cpr;

  auto item_ct = [&](int i, int64_t* c, int64_t* t) {
    *c = i / nt;
    *t = tlist[i - (int)(*c) * nt];
  };
  // TMA loader: lane 0 arms the stage's mbarrier and issues one tensor copy for the window.
  auto issue_tma = [&](int i, int s) {
    if (lane == 0) {
      int64_t c, t;
      item_ct(i, &c, &t);
      load_window(&tmap, p, p.unit, m, c, t, my_stage0 + s * p.stage_bytes, my_bar0 + s * 8, tx_bytes);
    }
  };
  // LSU loader: the warp streams the window's 16-byte chunks with cp.async (32-byte sector
  // granularity in L2/DRAM instead of the 128-byte lines TMA fetches); chunks that start right of
  // the image row or that the shifted row does not touch are skipped.
  auto issue_lsu = [&](int i, int s) {
    int64_t c, t;
    item_ct(i, &c, &t);
    const int32_t top = p.boxes[(m * p.T + t) * 2];
    const int32_t left_u = p.boxes[(m * p.T + t) * 2 + 1] * p.unit;
    const int left_al = left_u & ~7;
    const int last_chunk = ((left_u & 7) + p.wu - 1) >> 3;               // last chunk the row touches
    const int max_chunk = (int)((p.Wu - left_al) >> 3) - 1;              // last chunk inside the image row
    const int lim = last_chunk < max_chunk ? last_chunk : max_chunk;
    const uint16_t* base = p.image + ((c * p.T + t) * p.H + top) * p.Wu + left_al;
    const uint32_t dst0 = my_stage0 + s * p.stage_bytes;
    int row = lane / cpr, col = lane - row * cpr;
    const int drow = 32 / cpr, dcol = 32 - drow * cpr;
    for (int j = lane; j < n_chunks; j += 32) {
      if (col <= lim) cp_async16(dst0 + j * 16, base + (int64_t)row * p.Wu + col * 8);
      row += drow;
      col += dcol;
      if (col >= cpr) { col -= cpr; ++row; }
    }
  };

  if (p.loader == 0) {
    for (int s = 0; s < p.n_stages - 1; ++s) {
      const int i = warp + s * nw;
      if (i < n_items) issue_tma(i, s);
    }
  } else {
    for (int s = 0; s < p.n_stages - 1; ++s) {
      const int i = warp + s * nw;
      if (i < n_items) issue_lsu(i, s);
      cp_async_commit();
    }
  }
  int s = 0;
  uint32_t parity = 0;
  for (int i = warp; i < n_items; i += nw) {
    // refill the stage the previous item used (every lane is past reading it)
    {
      const int nxt = i + (p.n_stages - 1) * nw;
      int rs = s + p.n_stages - 1;
      if (rs >= p.n_stages) rs -= p.n_stages;
      if (p.loader == 0) {
        if (nxt < n_items) issue_tma(nxt, rs);
      } else {
        if (nxt < n_items) issue_lsu(nxt, rs);
        cp_async_commit();
      }
    }
    int64_t c, t;
    item_ct(i, &c, &t);
    const int shift = (p.boxes[(m * p.T + t) * 2 + 1] * p.unit) & 7;
    const int64_t n = (m * p.C + c) * p.T + t;
    uint16_t* dst = STORE ? p.roi + n * (int64_t)p.rows * p.wu : nullptr;
    const uint8_t* buf = my_stages + (size_t)s * p.stage_bytes;
    if (p.loader == 0) {
      mbar_wait(my_bar0 + s * 8, parity);
    } else {
      // all but the newest n_stages-1 groups are complete -> this item's chunks have landed
      switch (p.n_stages) {
        case 2: cp_async_wait<1>(); break;
        case 3: cp_async_wait<2>(); break;
        default: cp_async_wait<3>(); break;
      }
      __syncwarp();
    }
    uint32_t sf = 0, sb = 0;
    if (p.vpr) {
      switch (shift) {
#define MGB_CONSUME(SS) \
  case SS: consume_vec<STATS, STORE, SS, VPL>(p, buf, dst, fgm, bgm, lane, fm, bm, svo, &sf, &sb); break;
        MGB_CONSUME(0) MGB_CONSUME(1) MGB_CONSUME(2) MGB_CONSUME(3)
        MGB_CONSUME(4) MGB_CONSUME(5) MGB_CONSUME(6)
        default: consume_vec<STATS, STORE, 7, VPL>(p, buf, dst, fgm, bgm, lane, fm, bm, svo, &sf, &sb); break;
#undef MGB_CONSUME
      }
    } else {
      consume_generic<STATS, STORE>(p, buf, dst, fgm, bgm, lane, shift, &sf, &sb);
    }
    if constexpr (STATS) {
      sf = __reduce_add_sync(0xffffffffu, sf);
      sb = __reduce_add_sync(0xffffffffu, sb);
      write_stats(p, lane, n, cnt_fg, cnt_bg, (double)sf, (double)sb, nan_f64(), nan_f64());
    }
    __syncwarp();
    if (++s == p.n_stages) { s = 0; parity ^= 1; }
  }
}

// ---------------------------------------------------------------------------------------------
// Warp-per-marker variant for MANY markers with FEW windows each (bead screens: 1e5 markers x 48
// windows of 50x50).  With one CTA per marker the mask set-up, the block barrier and the pipeline
// fill are paid once per 48 windows and spread over 8 warps (6 windows each); here every warp owns
// a marker for all its windows, keeps the marker's mask bytes in registers and runs one long
// TMA pipeline -- no block-level synchronisation after the start.  Window rows that are not a
// whole number of 16-byte vectors (50 px = 100 B) are handled as 8-byte quads: the flat roi is
// 4-pixel aligned (L*L*2 is a multiple of 8 for even L), a quad is one or two pixel pairs of one or
// two window rows, each pair one or two aligned 32-bit shared-memory words funnel-shifted by the
// window's parity.  QPL = quads per lane (unrolled, offsets and masks in registers).
// ---------------------------------------------------------------------------------------------

template <bool STATS, bool STORE, int QPL>
__global__ void __launch_bounds__(kTmaMaxWarps * 32, 1)
roi_gather_wpm_kernel(const __grid_constant__ CUtensorMap tmap, const TmaGatherParams p, int64_t M) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nw = blockDim.x >> 5;
  const int tm = blockIdx.y;

  uint8_t* stages = smem;                                                  // [warp][stage][stage_bytes]
  uint64_t* bars = reinterpret_cast<uint64_t*>(stages + (size_t)nw * p.n_stages * p.stage_bytes);
  int32_t* tlist = reinterpret_cast<int32_t*>(bars + kTmaMaxWarps * 8);
  __shared__ int s_nt;
  if (warp == 0) {
    const int n = list_timepoints<STATS>(p, tm, tlist, lane);
    if (lane == 0) s_nt = n;
  }
  if (lane == 0) init_stage_barriers(&bars[warp * 8], p.n_stages);
  __syncthreads();
  const int64_t mi = (int64_t)blockIdx.x * nw + warp;
  if (mi >= M) return;
  const int64_t m = p.order ? p.order[mi] : mi;
  const int nt = s_nt;
  const int n_items = nt * (int)p.C;

  // window-independent per-lane state: for each quad its two pixel pairs' offsets in the staged
  // window (16-bit units, without the window's shift) and the 4+4 mask bytes
  const int nquads = (p.rows * p.wu) >> 2;
  uint32_t offa[QPL], offb[QPL], fm[QPL], bm[QPL];
  uint32_t nf = 0, nb = 0;
  const uint32_t* f32 = STATS ? reinterpret_cast<const uint32_t*>(p.fg + (m * p.Tm + tm) * (int64_t)p.rows * p.rows) : nullptr;
  const uint32_t* b32 = STATS ? reinterpret_cast<const uint32_t*>(p.bg + (m * p.Tm + tm) * (int64_t)p.rows * p.rows) : nullptr;
#pragma unroll
  for (int k = 0; k < QPL; ++k) {
    const int q = lane + 32 * k;
    const int u = q < nquads ? 4 * q : 0;
    const int row = u / p.wu, col = u - row * p.wu;
    offa[k] = row * p.wpu + col;
    offb[k] = (col + 2 < p.wu) ? offa[k] + 2 : (row + 1) * p.wpu;     // second pair wraps to the next row
    fm[k] = bm[k] = 0;
    if constexpr (STATS) {
      if (q < nquads) {
        // any non-zero byte counts as set (0/255 masks are as good as 0/1)
        fm[k] = __vcmpne4(__ldg(f32 + q), 0u) & 0x01010101u;
        bm[k] = __vcmpne4(__ldg(b32 + q), 0u) & 0x01010101u;
        nf += __popc(fm[k]);
        nb += __popc(bm[k]);
      }
    }
  }
  double cnt_fg = 0.0, cnt_bg = 0.0;
  if constexpr (STATS) {
    cnt_fg = (double)__reduce_add_sync(0xffffffffu, nf);
    cnt_bg = (double)__reduce_add_sync(0xffffffffu, nb);
  }

  uint8_t* my_stages = stages + (size_t)warp * p.n_stages * p.stage_bytes;
  const uint32_t my_stage0 = smem_u32(my_stages);
  const uint32_t my_bar0 = smem_u32(&bars[warp * 8]);
  const uint32_t tx_bytes = (uint32_t)(p.rows * p.wpu * 2);

  auto item_ct = [&](int i, int64_t* c, int64_t* t) {
    *c = i / nt;
    *t = tlist[i - (int)(*c) * nt];
  };
  auto issue_tma = [&](int i, int s) {
    if (lane == 0) {
      int64_t c, t;
      item_ct(i, &c, &t);
      load_window(&tmap, p, p.unit, m, c, t, my_stage0 + s * p.stage_bytes, my_bar0 + s * 8, tx_bytes);
    }
  };
  for (int s = 0; s < p.n_stages - 1; ++s)
    if (s < n_items) issue_tma(s, s);
  int s = 0;
  uint32_t parity = 0;
  for (int i = 0; i < n_items; ++i) {
    {
      const int nxt = i + p.n_stages - 1;
      int rs = s + p.n_stages - 1;
      if (rs >= p.n_stages) rs -= p.n_stages;
      if (nxt < n_items) issue_tma(nxt, rs);
    }
    int64_t c, t;
    item_ct(i, &c, &t);
    const uint32_t shift = (uint32_t)(p.boxes[(m * p.T + t) * 2 + 1] * p.unit) & 7u;
    const int64_t n = (m * p.C + c) * p.T + t;
    uint2* dst = STORE ? reinterpret_cast<uint2*>(p.roi + n * (int64_t)p.rows * p.wu) : nullptr;
    const uint32_t* s32 = reinterpret_cast<const uint32_t*>(my_stages + (size_t)s * p.stage_bytes);
    mbar_wait(my_bar0 + s * 8, parity);
    uint32_t sf = 0, sb = 0;
    auto consume = [&](auto par) {
      constexpr int PAR = decltype(par)::value;
#pragma unroll
      for (int k = 0; k < QPL; ++k) {
        const int q = lane + 32 * k;
        if (q < nquads) {
          const uint32_t lo = load_pair<PAR>(s32, offa[k] + shift);
          const uint32_t hi = load_pair<PAR>(s32, offb[k] + shift);
          if constexpr (STORE) {
            asm volatile("st.global.L1::no_allocate.v2.u32 [%0], {%1,%2};" ::"l"(dst + q), "r"(lo), "r"(hi) : "memory");
          }
          if constexpr (STATS) {
            sf = __dp2a_lo(lo, fm[k], sf); sf = __dp2a_hi(hi, fm[k], sf);
            sb = __dp2a_lo(lo, bm[k], sb); sb = __dp2a_hi(hi, bm[k], sb);
          }
        }
      }
    };
    if (shift & 1u) consume(std::integral_constant<int, 1>{});
    else consume(std::integral_constant<int, 0>{});
    if constexpr (STATS) {
      sf = __reduce_add_sync(0xffffffffu, sf);
      sb = __reduce_add_sync(0xffffffffu, sb);
      write_stats(p, lane, n, cnt_fg, cnt_bg, (double)sf, (double)sb, nan_f64(), nan_f64());
    }
    __syncwarp();
    if (++s == p.n_stages) { s = 0; parity ^= 1; }
  }
}

int g_gather_wpm = 1;      // warp-per-marker kernel for many-marker shapes (tuning switch)
int g_gather_loader = 0;   // 0 = TMA tensor copies (default), 1 = cp.async chunks; equal within 1% on B200

// Returns MGB_OK when launched, MGB_EALIGN when this path does not apply (caller falls back to
// the LSU kernels of roi.cu), or an error.
int roi_gather_tma(const GatherArgs& a, cudaStream_t st) {
  if (a.itemsize < 2) return MGB_EALIGN;
  StagedWindow w;
  const int rc = stage_window(a, w);
  if (rc != MGB_OK) return rc;
  TmaGatherParams& p = w.p;
  const int64_t M = a.M;
  const int L = a.L, wu = p.wu;
  const CopyLoop loop = choose_copy_loop(p, a.roi, false);
  const size_t mask_bytes = a.with_stats ? 2 * (size_t)((L * wu + 15) & ~15) : 0;
  const size_t fixed = mask_bytes + kTmaMaxWarps * 8 * sizeof(uint64_t) + (size_t)a.T * sizeof(int32_t) + 128;
  const size_t budget = (size_t)w.max_smem > fixed + 1024 ? (size_t)w.max_smem - fixed - 1024 : 0;
  int nw = kTmaMaxWarps;
  if (const char* e = getenv("MGB_GATHER_WARPS")) nw = atoi(e) == 4 ? 4 : kTmaMaxWarps;   // tuning only
  int ns = (int)(budget / ((size_t)nw * p.stage_bytes));
  if (ns < 2) {
    nw = 4;
    ns = (int)(budget / ((size_t)nw * p.stage_bytes));
  }
  if (ns > 4) ns = 4;
  if (ns < 2) return MGB_EALIGN;
  p.n_stages = ns;
  const size_t smem_bytes = (size_t)nw * ns * p.stage_bytes + fixed;
  p.loader = g_gather_loader;

  // Many markers, rows that are not whole 16-byte vectors, few quads per lane: warp-per-marker.
  const int qpl = ((L * wu) / 4 + 31) / 32;
  const bool masks_0_1_words = !a.with_stats || (((size_t)L * L) % 4 == 0 && (reinterpret_cast<uintptr_t>(a.fg) & 3u) == 0 &&
                                                 (reinterpret_cast<uintptr_t>(a.bg) & 3u) == 0);
  if (g_gather_wpm && p.unit == 1 && copy_loop(L, wu, a.roi, true) == CopyLoop::kQuad && M >= 2048 && masks_0_1_words) {
    const size_t fixed_w = kTmaMaxWarps * 8 * sizeof(uint64_t) + (size_t)a.T * sizeof(int32_t) + 128;
    const size_t budget_w = (size_t)w.max_smem > fixed_w + 1024 ? (size_t)w.max_smem - fixed_w - 1024 : 0;
    int ns_w = (int)(budget_w / ((size_t)kTmaMaxWarps * p.stage_bytes));
    if (ns_w > 4) ns_w = 4;
    if (ns_w >= 2) {
      TmaGatherParams pw = p;
      pw.n_stages = ns_w;
      const size_t smem_w = (size_t)kTmaMaxWarps * ns_w * p.stage_bytes + fixed_w;
      dim3 grid_w((unsigned)((M + kTmaMaxWarps - 1) / kTmaMaxWarps), (unsigned)p.Tm);
#define MGB_LAUNCH_W(ST, SO, QP)                                                                       \
  do {                                                                                                 \
    MGB_CUDA_TRY(cudaFuncSetAttribute(roi_gather_wpm_kernel<ST, SO, QP>,                               \
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_w));      \
    roi_gather_wpm_kernel<ST, SO, QP><<<grid_w, kTmaMaxWarps * 32, smem_w, st>>>(w.tmap, pw, M);       \
    record_gather_path(kGatherStagedWpm, QP, CopyLoop::kQuad, kTmaMaxWarps, ns_w, 0, ST, SO);           \
  } while (0)
#define MGB_LAUNCH_WQ(ST, SO)                      \
  do {                                             \
    if (qpl <= 12) MGB_LAUNCH_W(ST, SO, 12);       \
    else if (qpl <= 20) MGB_LAUNCH_W(ST, SO, 20);  \
    else MGB_LAUNCH_W(ST, SO, 24);                 \
  } while (0)
      if (a.with_stats) {
        if (a.roi) MGB_LAUNCH_WQ(true, true);
        else MGB_LAUNCH_WQ(true, false);
      } else {
        MGB_LAUNCH_WQ(false, true);
      }
#undef MGB_LAUNCH_WQ
#undef MGB_LAUNCH_W
      MGB_CUDA_LAUNCH_CHECK();
      return MGB_OK;
    }
  }
  const int vpl = p.vpr ? (int)((L * p.vpr + 31) / 32) : 0;       // vectors per lane
  dim3 grid((unsigned)M, (unsigned)p.Tm);
#define MGB_LAUNCH(ST, SO, VP)                                                                          \
  do {                                                                                                  \
    MGB_CUDA_TRY(cudaFuncSetAttribute(roi_gather_tma_kernel<ST, SO, VP>,                                \
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));   \
    roi_gather_tma_kernel<ST, SO, VP><<<grid, nw * 32, smem_bytes, st>>>(w.tmap, p);                    \
    record_gather_path(kGatherStagedCta, VP, loop, nw, ns, p.loader, ST, SO);                           \
  } while (0)
#define MGB_LAUNCH_V(ST, SO)                                  \
  do {                                                        \
    if (vpl > 0 && vpl <= 12) MGB_LAUNCH(ST, SO, 12);         \
    else if (vpl > 12 && vpl <= 21) MGB_LAUNCH(ST, SO, 21);   \
    else if (vpl > 21 && vpl <= 36) MGB_LAUNCH(ST, SO, 36);   \
    else MGB_LAUNCH(ST, SO, 0);                               \
  } while (0)
  if (a.with_stats) {
    if (a.roi) MGB_LAUNCH_V(true, true);
    else MGB_LAUNCH_V(true, false);
  } else {
    MGB_LAUNCH_V(false, true);
  }
#undef MGB_LAUNCH_V
#undef MGB_LAUNCH
  MGB_CUDA_LAUNCH_CHECK();
  return MGB_OK;
}

}  // namespace mgb
