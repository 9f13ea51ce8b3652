// Shared helpers for the magnify_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/magnify_b200.h"

// Every kernel launch of the library is followed by this macro: it counts the launch (the
// count is what bench.py reports as gpu_launches) and surfaces launch errors.
extern "C" void mgb_count_launch_(void);
#define MGB_CUDA_LAUNCH_CHECK()                      \
  do {                                               \
    mgb_count_launch_();                             \
    cudaError_t e__ = cudaGetLastError();            \
    if (e__ != cudaSuccess) return (int)e__;         \
  } while (0)

#define MGB_CUDA_TRY(expr)                           \
  do {                                               \
    cudaError_t e__ = (expr);                        \
    if (e__ != cudaSuccess) return (int)e__;         \
  } while (0)

namespace mgb {

constexpr int kThreads = 256;

__host__ __device__ inline bool aligned16(const void* p) {
  return (reinterpret_cast<uintptr_t>(p) & 15u) == 0;
}

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ceil(2^32 / d): the copy loops divide an index x by d as __umulhi(x, magic_u32(d)).  d = 1 has no
// 32-bit value, so a loop that divides by d is never chosen for d = 1.
inline uint32_t magic_u32(uint32_t d) { return (uint32_t)((0x100000000ULL + d - 1) / d); }

// Doubles per summary record of (marker, channel, time):
// n_fg, n_bg, sum_fg, sum_bg, mean_fg, mean_bg, median_fg, median_bg.
constexpr int kStatsRec = 8;

// Stream-ordered scratch for the few entry points whose temporary sizes are only known inside the
// call (CUB temp storage, the unique-circle list, large-mask workspaces).  The blocks come from a
// PRIVATE memory pool per device, created on first use, that keeps at most 1 GiB of freed blocks
// cached: repeated calls do not pay an allocation from the driver each time, and the process-wide
// default pool (which the caller's framework may rely on) is left exactly as it was.
inline cudaError_t scratch_alloc(void** ptr, size_t bytes, cudaStream_t stream) {
  static cudaMemPool_t pools[64] = {};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= 64) return cudaMallocAsync(ptr, bytes, stream);
  if (!pools[dev]) {
    cudaMemPoolProps props = {};
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = dev;
    cudaMemPool_t pool = nullptr;
    e = cudaMemPoolCreate(&pool, &props);
    if (e != cudaSuccess) return e;
    unsigned long long keep = 1ull << 30;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    pools[dev] = pool;
  }
  return cudaMallocFromPoolAsync(ptr, bytes, pools[dev], stream);
}

// Streaming 128-bit global accesses: every tile / image / roi byte is touched once per pass,
// so keep them out of L1 (the coefficient tables and masks are what should stay cached).
__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_stream(uint4* p, const uint4& v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x),
               "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}

__device__ __forceinline__ void atomic_max_nonneg_f64(double* addr, double v) {
  // Non-negative IEEE doubles order like their bit patterns.
  atomicMax(reinterpret_cast<unsigned long long*>(addr),
            static_cast<unsigned long long>(__double_as_longlong(v)));
}

__device__ __forceinline__ double nan_f64() { return __longlong_as_double(0x7ff8000000000000LL); }

// 8 consecutive 16-bit units starting S units into the 16 units of (a, b).
template <int S>
__device__ __forceinline__ uint4 shift_units(const uint4& a, const uint4& b) {
  const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  constexpr int o = S >> 1;
  if constexpr ((S & 1) == 0) {
    return make_uint4(w[o], w[o + 1], w[o + 2], w[o + 3]);
  } else {
    return make_uint4(__funnelshift_r(w[o], w[o + 1], 16), __funnelshift_r(w[o + 1], w[o + 2], 16),
                      __funnelshift_r(w[o + 2], w[o + 3], 16), __funnelshift_r(w[o + 3], w[o + 4], 16));
  }
}

// 16-byte global -> shared copy that bypasses L1 (cp.async.cg, SASS LDGSTS), and its completion:
// commit closes a group of copies, wait<N> returns once at most N groups are still in flight.
__device__ __forceinline__ void cp_async16(uint32_t smem_addr, const void* gptr) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(gptr) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

}  // namespace mgb
