// Host side of the fused pixel-text InfoNCE (rc_infonce_bf16 and its variants): workspace sizing, the pre-pass kernels
// (1/|x_p| and the bf16 copy of an fp32 X, optionally with the smoothness sums) and the dispatcher that validates the
// arguments, runs the pre-pass and launches one of the kernels:
//   dText   infonce_umma2.cu (writes G) + infonce_dt_umma.cu (dT = G^T X)
//   1-CTA   infonce_umma.cu   D = 128 / 384
//   TS      infonce_ts.cu     backward launches without dText, D = 256 / 512 / 768 / 1024 (rc_infonce_bf16_dyn's excepted)
//   SS      infonce_umma2.cu  forward-only launches, dText (D = 256 / 512), rc_infonce_bf16_dyn and RC_INFONCE_SS_KERNEL,
//                             D = 256 / 512 / 768 / 1024
#include "common.cuh"

extern "C" int64_t rc_infonce_workspace_bytes(int B, int D, int64_t HW, int K, rc_dtype x_dtype) {
  (void)K;
  const int64_t M = (int64_t)B * HW;
  int64_t bytes = ((M * 4 + 255) / 256) * 256;                                   // inv_norm
  if (x_dtype == RC_F32) bytes += (((int64_t)B * D * HW * 2 + 255) / 256) * 256;   // bf16 copy of X
  return bytes + 256;
}

extern "C" int64_t rc_infonce_workspace_bytes_dt(int B, int D, int64_t HW, int K, rc_dtype x_dtype) {
  const int64_t Kp = (K + 63) / 64 * 64;
  const int64_t base = (rc_infonce_workspace_bytes(B, D, HW, K, x_dtype) + 255) / 256 * 256;
  return base + (int64_t)B * HW * Kp * 2 + 512;       // + G, bf16 [B][HW][Kp]
}

namespace rc {

// ------------------------------------------------------------------------------------------------
// pre-pass: inverse row norms of the bf16-rounded rows (+ bf16 copy of an fp32 input)
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
rownorm_kernel(const T* __restrict__ x, int B, int D, int64_t HW, __nv_bfloat16* __restrict__ xb,
               float* __restrict__ inv_norm) {
  const int64_t groups_per_img = HW / 8;
  const int64_t n = (int64_t)B * groups_per_img;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n; g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = g / groups_per_img;
    const int64_t p0 = (g - b * groups_per_img) * 8;
    const T* src = x + b * (int64_t)D * HW + p0;
    __nv_bfloat16* dst = xb ? xb + b * (int64_t)D * HW + p0 : nullptr;
    float ss[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) ss[j] = 0.f;
    if (sizeof(T) == 2) {          // bf16 rows: nothing to round or copy, squares straight from the packed words
#pragma unroll 8
      for (int d = 0; d < D; ++d) {
        const uint4 w = __ldg(reinterpret_cast<const uint4*>(src + (int64_t)d * HW));
        const uint32_t u[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          ss[2 * j] = sqacc_bf16x2_lo(ss[2 * j], u[j]);
          ss[2 * j + 1] = sqacc_bf16x2_hi(ss[2 * j + 1], u[j]);
        }
      }
    } else
#pragma unroll 4
    for (int d = 0; d < D; ++d) {
      float v[8];
      load8(src + (int64_t)d * HW, v);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        v[j] = __bfloat162float(__float2bfloat16_rn(v[j]));   // the tensor cores see the rounded value
        ss[j] = fmaf(v[j], v[j], ss[j]);
      }
      if (dst) store8(dst + (int64_t)d * HW, v);
    }
    float o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = 1.f / fmaxf(sqrtf(ss[j]), 1e-12f);
    store8(inv_norm + b * HW + p0, o);
  }
}

// fp32 X: the same pre-pass AND the smoothness sums (tv.cu: sums[0] = sum |x[h][w+1] - x[h][w]|, sums[1] = sum |x[h+1][w] - x[h][w]|)
// from ONE read of X.  A thread owns a strip of R rows x 8 pixels and walks the channels; per channel it loads its R rows plus the
// row below (the only re-read: (R+1)/R of X, mostly L2 hits), takes the right-hand neighbour from the next lane (consecutive
// lanes = consecutive 8-pixel groups of the same rows), rounds to bf16 for the copy and the norms, and keeps the TV terms on
// the unrounded fp32 values as rc_tv_fwd does.  kCodes: the signs of those differences are kept as well -- 4 bits per element,
// one 32-bit word per 8-pixel group: pixel j at bits 4j..4j+3, low pair sgn(x[h][w] - x[h][w+1]), high pair
// sgn(x[h][w] - x[h+1][w]), each stored as sgn + 1 in two bits (0 / 1 / 2; 1 past the last column / row) -- which is all the
// smoothness BACKWARD needs (rc_tv_bwd_codes: 0.5 bytes per element read instead of x again).
constexpr int kPrepassTvRows = 4;      // R: rows per strip
constexpr int kPrepassTvThreads = 128;
constexpr int kPrepassTvBlocks = 4;    // resident blocks per SM (launch bounds)
constexpr int kPrepassTvUnroll = 1;    // channel-loop unroll
// acc + (sgn(d) + 1) * unit in FLOAT arithmetic, three FMA-pipe instructions per difference: d * 2^64 is normal for every
// non-zero d (an overflow to +-inf keeps its sign), so sat(d * 2^64 * 2^100 + 0.5) is exactly 0, 0.5 or 1 = (sgn(d) + 1) / 2.
// Four pixels x (horizontal, vertical) codes = 16 bits per accumulator: exact in a float.  (Packed bf16 compares of the
// differences -- set.gt/lt.bf16x2, two results per instruction --, integer selects and a two's-complement code from two
// saturating multiplies were measured too: 2.7-2.8 ms each, the pass is bound by its instruction count.)
__device__ __forceinline__ float add_sgn_code(float acc, float d, float unit) {
  const float q = __saturatef(fmaf(d * 18446744073709551616.f, 1.2676506002282294e30f, 0.5f));
  return fmaf(q, 2.f * unit, acc);
}

template <int R, bool kCodes>
__global__ void __launch_bounds__(kPrepassTvThreads, kPrepassTvBlocks)
rownorm_tv_kernel(const float* __restrict__ x, int B, int D, int H, int W, __nv_bfloat16* __restrict__ xb,
                  float* __restrict__ inv_norm, double* __restrict__ tv_sums, uint32_t* __restrict__ codes) {
  const int gpr = W >> 3;                                   // 8-pixel groups per row
  const int strips = (H + R - 1) / R;
  const int64_t HW = (int64_t)H * W;
  const int64_t n = (int64_t)B * strips * gpr;
  const int lane = threadIdx.x & 31;
  double acc_h = 0.0, acc_v = 0.0;
  for (int64_t u0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); u0 < n; u0 += (int64_t)gridDim.x * blockDim.x) {
    const bool live = u0 + lane < n;                        // warp-uniform trip count: dead lanes shadow the last unit, store nothing
    const int64_t u = live ? u0 + lane : n - 1;
    const int gi = (int)(u % gpr);
    const int64_t bs = u / gpr;
    const int strip = (int)(bs % strips);
    const int64_t b = bs / strips;
    const int h0 = strip * R;
    const int rows = min(R, H - h0);
    const bool has_below = h0 + rows < H;
    const bool has_right = gi + 1 < gpr;
    const bool right_shfl = has_right && lane < 31;         // lane + 1 then holds group gi + 1 of the same rows
    const int64_t off = b * (int64_t)D * HW + (int64_t)h0 * W + gi * 8;
    const float* src = x + off;
    __nv_bfloat16* dst = xb + off;
    uint32_t* cdst = kCodes ? codes + (b * (int64_t)D * H + h0) * gpr + gi : nullptr;
    float ss[R][8];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int j = 0; j < 8; ++j) ss[r][j] = 0.f;
#pragma unroll kPrepassTvUnroll
    for (int d = 0; d < D; ++d) {
      const float* p = src + (int64_t)d * HW;
      float v[R + 1][8];
#pragma unroll
      for (int r = 0; r <= R; ++r)
        if (r < rows || (r == rows && has_below)) load8(p + (int64_t)r * W, v[r]);
      float sh = 0.f, sv = 0.f;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        float right = __shfl_down_sync(0xffffffffu, v[r][0], 1);
        if (r < rows) {
          // a missing neighbour is replaced by the value itself: difference 0, sign code 0
          if (!right_shfl) right = has_right ? __ldg(p + (int64_t)r * W + 8) : v[r][7];
          const bool below = r + 1 < rows || has_below;
          uint32_t pk[4];
          float dh[8], dv[8];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            pk[i] = pack_bf16x2(v[r][2 * i], v[r][2 * i + 1]);                 // the tensor cores see the rounded value
            ss[r][2 * i] = sqacc_bf16x2_lo(ss[r][2 * i], pk[i]);
            ss[r][2 * i + 1] = sqacc_bf16x2_hi(ss[r][2 * i + 1], pk[i]);
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            dh[j] = v[r][j] - (j < 7 ? v[r][j + 1] : right);
            dv[j] = below ? v[r][j] - v[r + 1][j] : 0.f;
            sh += fabsf(dh[j]);
            sv += fabsf(dv[j]);
          }
          if (live) *reinterpret_cast<uint4*>(dst + (int64_t)d * HW + (int64_t)r * W) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          if (kCodes) {
            // word layout: pixel j at bits 4j..4j+3; +0 horizontal, +2 vertical
            float lo = 0.f, hi = 0.f;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              lo = add_sgn_code(add_sgn_code(lo, dh[j], (float)(1 << (4 * j))), dv[j], (float)(4 << (4 * j)));
              hi = add_sgn_code(add_sgn_code(hi, dh[j + 4], (float)(1 << (4 * j))), dv[j + 4], (float)(4 << (4 * j)));
            }
            if (live) cdst[((int64_t)d * H + r) * gpr] = __float2uint_rz(lo) | (__float2uint_rz(hi) << 16);
          }
        }
      }
      if (live) { acc_h += (double)sh; acc_v += (double)sv; }
    }
    if (live) {
#pragma unroll
      for (int r = 0; r < R; ++r)
        if (r < rows) {
          float o[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) o[j] = 1.f / fmaxf(sqrtf(ss[r][j]), 1e-12f);
          store8(inv_norm + b * HW + (int64_t)(h0 + r) * W + gi * 8, o);
        }
    }
  }
  acc_h = warp_sum(acc_h);
  acc_v = warp_sum(acc_v);
  __shared__ double red[2][kPrepassTvThreads / 32];
  if (lane == 0) { red[0][threadIdx.x >> 5] = acc_h; red[1][threadIdx.x >> 5] = acc_v; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, c = 0;
    for (int i = 0; i < kPrepassTvThreads / 32; ++i) { a += red[0][i]; c += red[1][i]; }
    atomicAdd(&tv_sums[0], a);
    atomicAdd(&tv_sums[1], c);
  }
}

int launch_rownorm_f32(const float* x, int B, int D, int64_t HW, __nv_bfloat16* xb, float* inv_norm, cudaStream_t s) {
  const int64_t blocks = ((int64_t)B * HW / 8 + 255) / 256;
  const int grid = (int)(blocks < (int64_t)num_sms() * 8 ? blocks : (int64_t)num_sms() * 8);
  rownorm_kernel<float><<<grid, 256, 0, s>>>(x, B, D, HW, xb, inv_norm);
  return check_launch("rownorm(f32 -> bf16)");
}
static int infonce_prepass_impl(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW, void* workspace,
                                int64_t workspace_bytes, cudaStream_t s, float** inv_norm_out, __nv_bfloat16** xb_out) {
  RC_REQUIRE(x && workspace, "rc_infonce_prepass: null pointer");
  if (HW % 8 != 0) return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16: HW=%lld must be a multiple of 8", (long long)HW);
  RC_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0, "rc_infonce_bf16: x must be 16-byte aligned");
  RC_REQUIRE(workspace_bytes >= rc_infonce_workspace_bytes(B, D, HW, 0, x_dtype), "rc_infonce_bf16: workspace too small");
  const int64_t M = (int64_t)B * HW;
  uint8_t* ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
  *inv_norm_out = reinterpret_cast<float*>(ws);
  *xb_out = (x_dtype == RC_F32) ? reinterpret_cast<__nv_bfloat16*>(ws + ((M * 4 + 255) / 256) * 256) : nullptr;
  if (s == (cudaStream_t)-1 || M == 0) return RC_OK;   // pointers only
  const int64_t groups = M / 8;
  const int64_t blocks = (groups + 255) / 256;
  const int grid = (int)(blocks < (int64_t)num_sms() * 8 ? blocks : (int64_t)num_sms() * 8);
  if (x_dtype == RC_F32) rownorm_kernel<float><<<grid, 256, 0, s>>>((const float*)x, B, D, HW, *xb_out, *inv_norm_out);
  else rownorm_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>((const __nv_bfloat16*)x, B, D, HW, nullptr, *inv_norm_out);
  return check_launch("rc_infonce_prepass");
}
}  // namespace rc

namespace rc { static long long* g_dbg_buf = nullptr; long long* debug_timing_buffer() { return g_dbg_buf; } }
#if defined(RC_BRINGUP) || defined(RC_TIMING)
extern "C" int rc_debug_set_timing_buffer(int64_t* dev_buf) { rc::g_dbg_buf = (long long*)dev_buf; return RC_OK; }
#endif

extern "C" int rc_infonce_prepass(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW, void* workspace,
                                  int64_t workspace_bytes, void* stream) {
  float* inv_norm; __nv_bfloat16* xb;
  int rcode = rc::check_sm100("rc_infonce_prepass");
  if (rcode) return rcode;
  return rc::infonce_prepass_impl(x, x_dtype, B, D, HW, workspace, workspace_bytes, (cudaStream_t)stream, &inv_norm, &xb);
}

// fp32 x [B][D][H][W], W % 8 == 0: the pre-pass of rc_infonce_bf16 (bf16 copy + 1/|x_p| into workspace, to be followed by
// RC_INFONCE_PREPASS_DONE) and the smoothness sums of rc_tv_fwd (ADDED to tv_sums[0..1]) from a single read of x; tv_codes
// (nullable, [B][D][H][W/8] words): the difference signs for rc_tv_bwd_codes.
extern "C" int rc_infonce_prepass_tv(const float* x, int B, int D, int H, int W, void* workspace, int64_t workspace_bytes,
                                     double* tv_sums, uint32_t* tv_codes, void* stream) {
  using namespace rc;
  RC_REQUIRE(x && workspace && tv_sums, "rc_infonce_prepass_tv: null pointer");
  RC_REQUIRE(B >= 0 && D >= 1 && H >= 0 && W >= 0, "rc_infonce_prepass_tv: bad shape");
  if (W % 8 != 0) return fail(RC_ERR_UNSUPPORTED, "rc_infonce_prepass_tv: W=%d must be a multiple of 8", W);
  int rcode = check_sm100("rc_infonce_prepass_tv");
  if (rcode) return rcode;
  const int64_t HW = (int64_t)H * W;
  float* inv_norm; __nv_bfloat16* xb;
  if ((rcode = infonce_prepass_impl(x, RC_F32, B, D, HW, workspace, workspace_bytes, (cudaStream_t)-1, &inv_norm, &xb))) return rcode;
  if (B == 0 || HW == 0) return RC_OK;
  constexpr int R = kPrepassTvRows;
  const int64_t units = (int64_t)B * ((H + R - 1) / R) * (W / 8);
  constexpr int T = kPrepassTvThreads;
  const int64_t blocks = (units + T - 1) / T;
  const int grid = (int)(blocks < (int64_t)num_sms() * 16 ? blocks : (int64_t)num_sms() * 16);
  if (tv_codes != nullptr) rownorm_tv_kernel<R, true><<<grid, T, 0, (cudaStream_t)stream>>>(x, B, D, H, W, xb, inv_norm, tv_sums, tv_codes);
  else rownorm_tv_kernel<R, false><<<grid, T, 0, (cudaStream_t)stream>>>(x, B, D, H, W, xb, inv_norm, tv_sums, nullptr);
  return check_launch("rc_infonce_prepass_tv");
}

// rep = 1: rc_infonce_bf16; rep = 4: rc_infonce_bf16_rep4 (y, w are [B*HW][4])
static int infonce_bf16_impl(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW, const void* t_bf16,
                             const void* tt_bf16, int K, const int32_t* y, const float* w, float inv_tau, float* lse,
                             double* loss_sum, double* w_sum, const double* w_sum_in, const float* grad_scale, void* dx,
                             float* dt, double* dlogtau, void* workspace, int64_t workspace_bytes, int flags, int rep,
                             void* stream, const int32_t* k_dev = nullptr, const float* log_tau_dev = nullptr,
                             bool dev_blocks = false, int k0 = 0) {
  using namespace rc;
  RC_REQUIRE(x && t_bf16 && y && w && workspace, "rc_infonce_bf16: null pointer");
  RC_REQUIRE(B >= 0 && HW >= 0, "rc_infonce_bf16: bad shape");
  if (K < 1 || K > 256) return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16: K=%d outside [1,256] (use rc_infonce_f32)", K);
  if (!(D == 128 || D == 384 || infonce_pair_supported(D)))
    return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16: D=%d must be 128, 256, 384, 512, 768 or 1024", D);
  RC_REQUIRE((reinterpret_cast<uintptr_t>(t_bf16) & 15) == 0, "rc_infonce_bf16: t must be 16-byte aligned");
  const bool bwd = dx != nullptr;
  if (bwd) RC_REQUIRE(tt_bf16 && w_sum_in && (reinterpret_cast<uintptr_t>(dx) & 15) == 0, "rc_infonce_bf16: backward needs tt_bf16, w_sum_in and aligned dx");
  if (dlogtau && !bwd) return fail(RC_ERR_INVALID, "rc_infonce_bf16: dlogtau needs dx");
  if (B == 0 || HW == 0) return RC_OK;
  int rcode = check_sm100("rc_infonce_bf16");
  if (rcode) return rcode;
  // CTA-pair kernels (cta_group::2) when the channel count allows it, the single-CTA kernel at D = 128 / 384.  The pair
  // kernels compute 1/|x_p| themselves from the operand tiles in shared memory, so a bf16 input needs no pre-pass at all
  // (an fp32 input still needs its bf16 copy).
  const bool use_pair = infonce_pair_supported(D);
  if ((k_dev != nullptr || log_tau_dev != nullptr) && !use_pair)
    return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16_dyn: device-side K / log tau need D = 256, 512, 768 or 1024 (CTA-pair kernel)");
  // rc_infonce_bf16_dyn_kblock: y is relative to k0 and w = 0 marks an ignored target, the RC_INFONCE_KEEP_WEIGHT form
  const int keep_w = (dev_blocks || (flags & RC_INFONCE_KEEP_WEIGHT)) ? 1 : 0;
  const int acc_dx = (flags & RC_INFONCE_ACCUMULATE_DX) ? 1 : 0;
  const float* lse_in = (flags & RC_INFONCE_LSE_GIVEN) ? lse : nullptr;
  if (acc_dx) RC_REQUIRE(bwd, "rc_infonce_bf16: RC_INFONCE_ACCUMULATE_DX needs dx");
  if (keep_w || lse_in || acc_dx) {      // rep = 1 or 4 (rc_infonce_bf16_dyn rejects these flags before it gets here)
    if (!use_pair || dt != nullptr)
      return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16: the K-blocked flags need D = 256, 512, 768 or 1024 and no dText");
    RC_REQUIRE(!(flags & RC_INFONCE_LSE_GIVEN) || lse != nullptr, "rc_infonce_bf16: RC_INFONCE_LSE_GIVEN needs lse");
  }
  if (rep != 1) {
    if (!use_pair) return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16_rep4: D=%d must be 256 or 512 (or 768 / 1024)", D);
    RC_REQUIRE((reinterpret_cast<uintptr_t>(y) & 15) == 0 && (reinterpret_cast<uintptr_t>(w) & 15) == 0,
               "rc_infonce_bf16_rep4: y and w must be 16-byte aligned");
  }
  if (dt != nullptr) {
    // the dText GEMM keeps all channels of a text row in the 512 tensor-memory columns of one CTA pair
    if (!use_pair || !bwd || D > 512)
      return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16: dText needs dx and D = 256 or 512 (use rc_infonce_f32 otherwise)");
    RC_REQUIRE(workspace_bytes >= rc_infonce_workspace_bytes_dt(B, D, HW, K, x_dtype), "rc_infonce_bf16: workspace too small for dText");
  }

  cudaStream_t s = (cudaStream_t)stream;
  float* inv_norm; __nv_bfloat16* xb;
  const bool skip_prepass = (flags & RC_INFONCE_PREPASS_DONE) || (use_pair && x_dtype == RC_BF16);
  if ((rcode = infonce_prepass_impl(x, x_dtype, B, D, HW, workspace, workspace_bytes, skip_prepass ? (cudaStream_t)-1 : s,
                                    &inv_norm, &xb))) return rcode;
  const void* xsrc = (x_dtype == RC_F32) ? (const void*)xb : x;
  if (!use_pair)
    return launch_infonce_1cta(xsrc, dx, t_bf16, tt_bf16, B, D, HW, K, inv_norm, y, w, inv_tau, grad_scale, w_sum_in, lse,
                               loss_sum, w_sum, dlogtau, s);
  InfoncePairArgs a{xsrc, dx, t_bf16, tt_bf16, B, D, HW, K, y, w, inv_tau, grad_scale, w_sum_in, lse, loss_sum, w_sum, dlogtau,
                    rep, keep_w, acc_dx, /*kb*/ 0, lse_in, /*g_out*/ nullptr, k_dev, log_tau_dev, k0};
  if (dt != nullptr) {
    // dText: the pair kernel also writes G = rs (P - sum onehot) (bf16 [B][HW][Kp]) into the workspace, then one
    // split-K GEMM over the pixels (infonce_dt_umma.cu) adds G^T X to dt.
    const int64_t base = rc_infonce_workspace_bytes(B, D, HW, K, x_dtype);
    uint8_t* ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
    a.g_out = ws + ((base + 255) / 256) * 256;
    if ((rcode = launch_infonce_pair(a, s))) return rcode;
    return launch_infonce_dt(a.g_out, xsrc, B, D, HW, K, dt, s);
  }
  // backward launches: the softmax tile as a tensor-memory operand of the dX GEMM (infonce_ts.cu) unless RC_INFONCE_SS_KERNEL;
  // the one-launch device-parameter form (rc_infonce_bf16_dyn) runs the SS kernel
  if (bwd && !(flags & RC_INFONCE_SS_KERNEL) && (dev_blocks || (k_dev == nullptr && log_tau_dev == nullptr)))
    return launch_infonce_ts(a, s);
  return launch_infonce_pair(a, s);
}

extern "C" int rc_infonce_bf16(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW, const void* t_bf16,
                               const void* tt_bf16, int K, const int32_t* y, const float* w, float inv_tau, float* lse,
                               double* loss_sum, double* w_sum, const double* w_sum_in, const float* grad_scale, void* dx,
                               float* dt, double* dlogtau, void* workspace, int64_t workspace_bytes, int flags, void* stream) {
  return infonce_bf16_impl(x, x_dtype, B, D, HW, t_bf16, tt_bf16, K, y, w, inv_tau, lse, loss_sum, w_sum, w_sum_in, grad_scale,
                           dx, dt, dlogtau, workspace, workspace_bytes, flags, 1, stream);
}

extern "C" int rc_infonce_bf16_rep4(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW, const void* t_bf16,
                                    const void* tt_bf16, int K, const int32_t* y4, const float* w4, float inv_tau, float* lse,
                                    double* loss_sum, double* w_sum, const double* w_sum_in, const float* grad_scale,
                                    void* dx, float* dt, double* dlogtau, void* workspace, int64_t workspace_bytes,
                                    int flags, void* stream) {
  return infonce_bf16_impl(x, x_dtype, B, D, HW, t_bf16, tt_bf16, K, y4, w4, inv_tau, lse, loss_sum, w_sum, w_sum_in,
                           grad_scale, dx, dt, dlogtau, workspace, workspace_bytes, flags, 4, stream);
}

// rep = 1 or 4; the number of valid candidate rows (<= K, the rest are zero pad rows) and log(tau) come from device memory
extern "C" int rc_infonce_bf16_dyn(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW, const void* t_bf16,
                                   const void* tt_bf16, int K, const int32_t* k_dev, const int32_t* y, const float* w,
                                   const float* log_tau_dev, int rep, float* lse, double* loss_sum, double* w_sum,
                                   const double* w_sum_in, const float* grad_scale, void* dx, double* dlogtau,
                                   void* workspace, int64_t workspace_bytes, int flags, void* stream) {
  RC_REQUIRE(log_tau_dev != nullptr, "rc_infonce_bf16_dyn: log_tau_dev is required");
  RC_REQUIRE(rep == 1 || rep == 4, "rc_infonce_bf16_dyn: rep must be 1 or 4");
  RC_REQUIRE(!(flags & (RC_INFONCE_KEEP_WEIGHT | RC_INFONCE_LSE_GIVEN | RC_INFONCE_ACCUMULATE_DX)), "rc_infonce_bf16_dyn: K-blocked flags are not supported");
  return infonce_bf16_impl(x, x_dtype, B, D, HW, t_bf16, tt_bf16, K, y, w, 0.f, lse, loss_sum, w_sum, w_sum_in, grad_scale, dx,
                           nullptr, dlogtau, workspace, workspace_bytes, flags, rep, stream, k_dev, log_tau_dev);
}

// rc_infonce_bf16_dyn for one block of the K-blocked rounds: rows [k0, k0 + K) of a contrast set whose valid row count is
// *k_dev; a launch whose block holds no valid row returns at once in the kernel (rangeclip_b200.h)
extern "C" int rc_infonce_bf16_dyn_kblock(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW, const void* t_bf16,
                                          const void* tt_bf16, int K, const int32_t* k_dev, int k0, const int32_t* y,
                                          const float* w, const float* log_tau_dev, int rep, float* lse, double* loss_sum,
                                          double* w_sum, const double* w_sum_in, const float* grad_scale, void* dx,
                                          double* dlogtau, void* workspace, int64_t workspace_bytes, int flags, void* stream) {
  using namespace rc;
  RC_REQUIRE(k_dev != nullptr && log_tau_dev != nullptr, "rc_infonce_bf16_dyn_kblock: k_dev and log_tau_dev are required");
  RC_REQUIRE(rep == 1 || rep == 4, "rc_infonce_bf16_dyn_kblock: rep must be 1 or 4");
  RC_REQUIRE(k0 >= 0, "rc_infonce_bf16_dyn_kblock: k0=%d must be >= 0", k0);
  if (K < 1 || K > 256) return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16_dyn_kblock: K=%d outside [1,256] (one block)", K);
  if (!infonce_pair_supported(D)) return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16_dyn_kblock: D=%d must be 256 or 512 (or 768 / 1024)", D);
  return infonce_bf16_impl(x, x_dtype, B, D, HW, t_bf16, tt_bf16, K, y, w, 0.f, lse, loss_sum, w_sum, w_sum_in, grad_scale, dx,
                           nullptr, dlogtau, workspace, workspace_bytes, flags, rep, stream, k_dev, log_tau_dev, true, k0);
}

extern "C" int rc_infonce_bf16_kblocks(const void* x, rc_dtype x_dtype, int D, int64_t HW, const void* t_bf16_all,
                                       const void* tt_bf16_all, int K, int n_blocks, const int32_t* y_rel, const float* w_rep,
                                       float inv_tau, float* lse, double* loss_sum, double* w_sum, const double* w_sum_in,
                                       const float* grad_scale, void* dx_blocks, double* dlogtau, void* workspace,
                                       int64_t workspace_bytes, int flags, void* stream) {
  using namespace rc;
  RC_REQUIRE(x && t_bf16_all && y_rel && w_rep && workspace && lse, "rc_infonce_bf16_kblocks: null pointer");
  RC_REQUIRE(HW >= 0 && K >= 1 && n_blocks >= 1 && n_blocks == (K + 255) / 256, "rc_infonce_bf16_kblocks: n_blocks must be ceil(K / 256)");
  if (!infonce_pair_supported(D)) return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16_kblocks: D=%d must be 256 or 512 (or 768 / 1024)", D);
  if (HW % 256 != 0) return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16_kblocks: HW=%lld must be a multiple of 256", (long long)HW);
  RC_REQUIRE((reinterpret_cast<uintptr_t>(t_bf16_all) & 15) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0, "rc_infonce_bf16_kblocks: alignment");
  const bool bwd = dx_blocks != nullptr;
  if (bwd) RC_REQUIRE(tt_bf16_all && w_sum_in && (flags & RC_INFONCE_LSE_GIVEN), "rc_infonce_bf16_kblocks: the backward needs tt_bf16_all, w_sum_in and RC_INFONCE_LSE_GIVEN");
  if (HW == 0) return RC_OK;
  int rcode = check_sm100("rc_infonce_bf16_kblocks");
  if (rcode) return rcode;
  cudaStream_t s = (cudaStream_t)stream;
  float* inv_norm; __nv_bfloat16* xb;
  const bool skip_prepass = (flags & RC_INFONCE_PREPASS_DONE) || x_dtype == RC_BF16;
  if ((rcode = infonce_prepass_impl(x, x_dtype, 1, D, HW, workspace, workspace_bytes, skip_prepass ? (cudaStream_t)-1 : s, &inv_norm, &xb))) return rcode;
  const void* xsrc = (x_dtype == RC_F32) ? (const void*)xb : x;
  const float* lse_in = (flags & RC_INFONCE_LSE_GIVEN) ? lse : nullptr;
  // the kb blocks of 256 candidate rows are the "images" of one launch; every target keeps its weight
  const InfoncePairArgs a{xsrc, dx_blocks, t_bf16_all, tt_bf16_all, n_blocks, D, HW, K, y_rel, w_rep, inv_tau, grad_scale,
                          w_sum_in, lse, loss_sum, w_sum, dlogtau, /*rep*/ 1, /*keep_w*/ 1, /*acc_dx*/ 0, /*kb*/ n_blocks, lse_in,
                          nullptr, nullptr, nullptr, 0};
  if (bwd && !(flags & RC_INFONCE_SS_KERNEL)) return launch_infonce_ts(a, s);
  return launch_infonce_pair(a, s);
}
