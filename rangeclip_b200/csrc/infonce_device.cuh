// Device helpers shared by the fused InfoNCE kernels (infonce_umma.cu, infonce_umma2.cu, infonce_ts.cu).
#pragma once
#include <stdint.h>

namespace rc {

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// r[i] for a per-thread dynamic i (registers cannot be indexed dynamically): binary select tree
__device__ __forceinline__ float select16(const uint32_t (&r)[16], int i) {
  float a[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] = __uint_as_float((i & 1) ? r[2 * j + 1] : r[2 * j]);
#pragma unroll
  for (int j = 0; j < 4; ++j) a[j] = (i & 2) ? a[2 * j + 1] : a[2 * j];
#pragma unroll
  for (int j = 0; j < 2; ++j) a[j] = (i & 4) ? a[2 * j + 1] : a[2 * j];
  return (i & 8) ? a[1] : a[0];
}

// Timing build (-DRC_TIMING, tools/timing*.py): per-role wait cycles, wt[tag] += cycles spent in the wait with that tag
// (wt[0] = lifetime), and an event trace of cluster 0.  The plain build compiles all of it away.
#ifdef RC_TIMING
__device__ __forceinline__ unsigned long long globaltimer_ns() {     // one clock for both CTAs of a pair
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define RC_T0(name) const long long name = clock64()
#define RC_TACC(idx, name) wt[idx] += clock64() - name
#define RC_WAIT(fn, bar, par, tag) do { const long long t0_ = clock64(); fn(bar, par, tag); wt[tag] += clock64() - t0_; } while (0)
// %globaltimer of event `id` of tile-pair iteration `iter` in [40, 44)
#define RC_EV(iter, id) do { if (prm.dbg != nullptr && blockIdx.x < 2 && lane == 0 && (iter) >= 40u && (iter) < 44u) \
    prm.dbg[256 + blockIdx.x * 192 + ((iter) - 40u) * 48 + (id)] = (long long)globaltimer_ns(); } while (0)
// a device function with RC_WAIT inside takes the caller's counters: f(... RC_WT_PARAM) called as f(... RC_WT)
#define RC_WT_PARAM , long long (&wt)[16]
#define RC_WT , wt
#else
#define RC_T0(name)
#define RC_TACC(idx, name)
#define RC_WAIT(fn, bar, par, tag) fn(bar, par, tag)
#define RC_EV(iter, id)
#define RC_WT_PARAM
#define RC_WT
#endif

}  // namespace rc
