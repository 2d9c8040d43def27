// Shared host/device helpers for the rangeclip_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <atomic>

#include "../../include/rangeclip_b200.h"

namespace rc {

// ---- error plumbing (no exceptions across the ABI) -------------------------------------------
extern thread_local char g_err[512];
extern std::atomic<long long> g_launches;

inline int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

inline int check_launch(const char* what) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(RC_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  return RC_OK;
}

#define RC_REQUIRE(cond, ...) \
  do { if (!(cond)) return ::rc::fail(RC_ERR_INVALID, __VA_ARGS__); } while (0)

inline int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

// the tensor-core kernels need an sm_100 device
inline int check_sm100(const char* what) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return fail(RC_ERR_NO_DEVICE, "%s: no CUDA device", what);
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (major != 10) return fail(RC_ERR_NO_DEVICE, "%s: needs an sm_100 device (compute capability %d.x found)", what, major);
  return RC_OK;
}

// fp32 -> bf16 copy + inverse row norms (defined in infonce.cu, shared with eval_topk_umma.cu)
int launch_rownorm_f32(const float* x, int B, int D, int64_t HW, __nv_bfloat16* xb, float* inv_norm, cudaStream_t s);

long long* debug_timing_buffer();   // bring-up instrumentation target (rc_debug_set_timing_buffer)
// The fused InfoNCE kernels; infonce.cu validates the arguments, runs the pre-pass and picks one of them.
// single-CTA version (infonce_umma.cu): D = 128 / 384, and the A/B baseline of the bring-up build
int launch_infonce_1cta(const void* xsrc, void* dx, const void* t_bf16, const void* tt_bf16, int B, int D, int64_t HW, int K,
                        const float* inv_norm, const int32_t* y, const float* w, float inv_tau, const float* grad_scale,
                        const double* w_sum_in, float* lse, double* loss_sum, double* w_sum, double* dlogtau, cudaStream_t s);
// CTA-pair (cta_group::2) versions of the fused InfoNCE kernel, D = 256 / 512: SS (infonce_umma2.cu, both dX operands in
// shared memory) and TS (infonce_ts.cu, the softmax tile as a tensor-memory operand); infonce_pair.cuh holds what they share
bool infonce_pair_supported(int D);
struct InfoncePairArgs {
  const void* xsrc;             // bf16 X [B][D][HW] (kb > 0: one image)
  void* dx;                     // bf16 dX [B][D][HW], null: forward only
  const void* t_bf16;           // T [Kall][D]
  const void* tt_bf16;          // T^T [D][Kall] (backward)
  int B, D;
  int64_t HW;
  int K;
  const int32_t* y;
  const float* w;
  float inv_tau;
  const float* grad_scale;
  const double* w_sum_in;
  float* lse;
  double* loss_sum;
  double* w_sum;
  double* dlogtau;
  int rep;                      // targets per row: 1, or 4 (the shared 2x2 form)
  int keep_w, acc_dx, kb;       // K-blocked launches (see cta_pair::Tiling)
  const float* lse_in;
  // SS only
  void* g_out;                  // dText: G = rs (P - sum onehot), bf16 [B][HW][Kp]
  // rc_infonce_bf16_dyn (SS) and rc_infonce_bf16_dyn_kblock (SS forward, TS backward): valid candidate rows and log tau in
  // device memory; k0 = the first contrast row of a K-blocked launch's block
  const int32_t* k_dev;
  const float* log_tau_dev;
  int k0;
};
int launch_infonce_pair(const InfoncePairArgs& a, cudaStream_t s);
// backward launches without dText, with host-side K and tau, or K-blocked with device-side K and tau
int launch_infonce_ts(const InfoncePairArgs& a, cudaStream_t s);
// dText = G^T X on the tensor cores (infonce_dt_umma.cu); G is the bf16 [B][HW][Kp] tensor the pair kernel writes
int launch_infonce_dt(const void* g, const void* xsrc, int B, int D, int64_t HW, int K, float* dt, cudaStream_t s);

// ---- device helpers ---------------------------------------------------------------------------
template <typename T> struct ElemIO;
template <> struct ElemIO<float> {
  static __device__ __forceinline__ float ld(const float* p) { return __ldg(p); }
  static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
};
template <> struct ElemIO<__nv_bfloat16> {
  static __device__ __forceinline__ float ld(const __nv_bfloat16* p) {
    return __bfloat162float(*p);
  }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
};

// Mixed-precision scalar arithmetic on the halves of a packed bf16x2 word (PTX fma/add .f32.bf16, SASS FHFMA.BF16 /
// FHADD.BF16 with .H0/.H1 operand selectors): the bf16 operand is widened inside the instruction, so there is no unpack
// instruction, and the result is the correctly rounded fp32 value -- bit-identical to unpack + FFMA / FADD.
__device__ __forceinline__ float sqacc_bf16x2_lo(float acc, uint32_t u) {      // acc + lo(u)^2
  float r;
  asm("{.reg .b16 lo, hi; mov.b32 {lo, hi}, %1; fma.rn.f32.bf16 %0, lo, lo, %2;}" : "=f"(r) : "r"(u), "f"(acc));
  return r;
}
__device__ __forceinline__ float sqacc_bf16x2_hi(float acc, uint32_t u) {      // acc + hi(u)^2
  float r;
  asm("{.reg .b16 lo, hi; mov.b32 {lo, hi}, %1; fma.rn.f32.bf16 %0, hi, hi, %2;}" : "=f"(r) : "r"(u), "f"(acc));
  return r;
}
__device__ __forceinline__ float addacc_bf16x2_lo(float acc, uint32_t u) {     // acc + lo(u)
  float r;
  asm("{.reg .b16 lo, hi; mov.b32 {lo, hi}, %1; add.rn.f32.bf16 %0, lo, %2;}" : "=f"(r) : "r"(u), "f"(acc));
  return r;
}
__device__ __forceinline__ float addacc_bf16x2_hi(float acc, uint32_t u) {     // acc + hi(u)
  float r;
  asm("{.reg .b16 lo, hi; mov.b32 {lo, hi}, %1; add.rn.f32.bf16 %0, hi, %2;}" : "=f"(r) : "r"(u), "f"(acc));
  return r;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// 8 consecutive elements -> floats (16B for bf16, 2x16B for f32); pointer must be 16B aligned.
__device__ __forceinline__ void load8(const float* p, float (&v)[8]) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p));
  const float4 b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void load8(const __nv_bfloat16* p, float (&v)[8]) {
  const uint4 r = __ldg(reinterpret_cast<const uint4*>(p));
  const uint32_t u[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = __uint_as_float(u[i] << 16);
    v[2 * i + 1] = __uint_as_float(u[i] & 0xffff0000u);
  }
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ void store8(float* p, const float (&v)[8]) {
  // one 256-bit store = one full 32-byte sector per lane; two 16-byte stores (stride 32 B across the warp) reach L2
  // as half-sector writes and halve the write bandwidth of store-only kernels
  if ((reinterpret_cast<uintptr_t>(p) & 31) == 0) {
    asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
                 "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                 : "memory");
  } else {
    reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
    reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
  }
}
__device__ __forceinline__ void store8(__nv_bfloat16* p, const float (&v)[8]) {
  uint4 r;
  r.x = pack_bf16x2(v[0], v[1]); r.y = pack_bf16x2(v[2], v[3]);
  r.z = pack_bf16x2(v[4], v[5]); r.w = pack_bf16x2(v[6], v[7]);
  *reinterpret_cast<uint4*>(p) = r;
}

}  // namespace rc
