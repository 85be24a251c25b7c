// Shared host/device helpers for liblbt_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "../../include/lbt.h"

namespace lbt {

// ---- host-side bookkeeping -------------------------------------------------------------------
extern std::atomic<uint64_t> g_launches;
void set_cuda_error(cudaError_t e, const char* where);

struct DeviceInfo {
  int device = -1;
  int sm_count = 0;
  int cc_major = 0, cc_minor = 0;
  bool ok = false;
};
// Immutable per-device cache (SM count, arch check).  Thread-safe.
const DeviceInfo& device_info();

inline int check_launch(const char* where) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_cuda_error(e, where);
    return LBT_ECUDA;
  }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return LBT_OK;
}

// ---- programmatic dependent launch (PDL) ------------------------------------------------------------------------
// A training step is ~140 short kernels back to back.  Launched with the programmatic-serialization attribute, kernel
// N+1 is scheduled while kernel N drains: its prologue (barrier init, TMEM allocation, tables) overlaps N's tail and it
// blocks at pdl_wait() — before its first global-memory access — until N has completed and flushed.  Captured into the
// step's CUDA graph as programmatic edges.  lbt_set_pdl(0) turns the attribute off (plain stream order).
extern std::atomic<int> g_pdl;
// Shared-memory carveout preference (percent, -1 = leave the driver's heuristic) applied to every kernel launched through
// launch_pdl: consecutive kernels that want different L1 / shared-memory splits force the SM to drain and reconfigure
// between them, and cannot overlap under programmatic dependent launch.  lbt_set_carveout() / LBT_CARVEOUT.
extern std::atomic<int> g_carveout;
void apply_carveout(const void* kernel);

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  apply_carveout(reinterpret_cast<const void*>(kernel));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = g_pdl.load(std::memory_order_relaxed) ? 1 : 0;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// n / d for runtime-constant d without the ~25-instruction integer division: q = umulhi(n, mul) >> shr, valid for n < 2^31
// (CUTLASS FastDivmod).  Host: make_fastdiv(d); device: fastdiv(n, fd), fastmod via n - q*d.
struct FastDiv {
  uint32_t d, mul, shr;
};
inline FastDiv make_fastdiv(uint32_t d) {
  FastDiv f{d, 0u, 0u};
  if (d > 1) {
    uint32_t lg = 0;
    while ((1ull << lg) < d) ++lg;
    const uint32_t pw = 31 + lg;
    f.mul = (uint32_t)(((1ull << pw) + d - 1) / d);
    f.shr = pw - 32;
  }
  return f;
}

// Most products one s32 accumulator may sum exactly for operand kinds a, b (LBT_MANT_*): |s8*s8| <= 2^14 and |u8*s8| <= 255*128,
// so 65536 of them stay below 2^31; |u8*u8| <= 255^2 allows only 32768 (2^15 * 65025 < 2^31 - 1 < 2^16 * 65025).
inline uint32_t max_products(int a_kind, int b_kind) {
  return (a_kind == LBT_MANT_U8 && b_kind == LBT_MANT_U8) ? 32768u : 65536u;
}

#define LBT_REQUIRE_ARCH()                        \
  do {                                            \
    const ::lbt::DeviceInfo& _di = ::lbt::device_info(); \
    if (!_di.ok) return _di.device < 0 ? LBT_ECUDA : LBT_EARCH; \
  } while (0)

// ---- device helpers --------------------------------------------------------------------------
#ifdef __CUDACC__

// Everything a kernel reads or writes in global memory must come after pdl_wait(); pdl_trigger() lets the next
// kernel of the stream start being scheduled (it still waits for this grid's completion at its own pdl_wait()).
__device__ __forceinline__ uint32_t fastdiv(uint32_t n, const FastDiv& f) { return f.d == 1 ? n : (__umulhi(n, f.mul) >> f.shr); }

#ifndef LBT_PDL_TRIGGER_AFTER_WAIT
#define LBT_PDL_TRIGGER_AFTER_WAIT 1
#endif
// LBT_PDL_TRIGGER_AFTER_WAIT = 1: a kernel lets its successor start only once its OWN wait has returned, i.e. once its
// predecessor has completed.  By induction everything older than the immediate predecessor is then complete when a kernel
// starts, so data produced two or more launches earlier (the packed weights of lbt_param_prep) may be read BEFORE the wait.
__device__ __forceinline__ void pdl_wait() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
#if LBT_PDL_TRIGGER_AFTER_WAIT
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
}
__device__ __forceinline__ void pdl_trigger() {
#if !LBT_PDL_TRIGGER_AFTER_WAIT
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
}

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

// u in [0, 1 - 2^-24]: the top 24 bits of a 32-bit draw.
__device__ __forceinline__ float u01(uint32_t r) { return __uint2float_rn(r >> 8) * 5.9604644775390625e-08f; }

// Noise for inner indices 4g .. 4g+3.
__device__ __forceinline__ float4 philox_noise4(uint64_t g, uint64_t seed, uint64_t off) {
  const uint4 r = philox4x32_10(make_uint4((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)off, (uint32_t)(off >> 32)),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  return make_float4(u01(r.x), u01(r.y), u01(r.z), u01(r.w));
}

__device__ __forceinline__ float4 ld_stream_f4(const float* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}

__device__ __forceinline__ uint32_t warp_sum(uint32_t v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// 2^e as an exact fp32 (e clamped to the normal range).
__device__ __forceinline__ float exp2i(int e) {
  e = max(-126, min(127, e));
  return __int_as_float((e + 127) << 23);
}

#endif  // __CUDACC__

}  // namespace lbt
