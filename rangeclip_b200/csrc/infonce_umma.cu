// K1/K2: fused pixel-text InfoNCE forward + backward on the 5th-gen tensor cores (sm_100a).
//
// Replaces model.py:272-291 (normalize, [N,512]@[512,K], /tau, cross_entropy) and its autograd
// (CE backward, two matmuls, normalize backward, index_put/scatter_add) with
//   * rownorm_kernel      one pass over X: 1/|x_p| (and the bf16 copy when X is fp32)
//   * infonce_umma_kernel persistent, warp-specialised: per 128-pixel tile
//        S  = X^T T^T           tcgen05.mma, A = X tile straight from NCHW (MN-major via TMA),
//                               B = text rows (K-major via TMA), fp32 accumulators in TMEM
//        softmax/CE epilogue    one thread per pixel reads its S row from TMEM: logsumexp, loss,
//                               dlogtau, and P = exp(z-m) - sum*onehot written as bf16 to smem
//        dX^T = T^T P^T          tcgen05.mma per 128-channel block, accumulators in TMEM
//        dX epilogue            row scale + normalize-backward projection, TMA store to NCHW
//     The [B*HW, K] logits never leave the SM.
//   * infonce_dt_umma_kernel  dText = P^T Xhat, text rows sliced across CTAs, S recomputed
//                             slice-wise from the saved logsumexp (TMEM cannot hold S, dX and the
//                             256x512 fp32 dText at once).
#include "common.cuh"
#include "umma.cuh"
#include <float.h>
#include <stdlib.h>

namespace rc {

using namespace umma;

// ------------------------------------------------------------------------------------------------
// host: driver entry point + tensor maps
// ------------------------------------------------------------------------------------------------
PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (PFN_encodeTiled)p;
  }
  return fn;
}

int make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box, const char* what) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return fail(RC_ERR_NO_DEVICE, "%s: cuTensorMapEncodeTiled entry point unavailable", what);
  cuuint64_t gdim[3];
  cuuint64_t gstr[2];
  cuuint32_t bx[3];
  cuuint32_t es[3] = {1, 1, 1};
  for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; }
  for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i + 1];
  const CUtensorMapSwizzle sw = (box[0] * 2 >= 128) ? CU_TENSOR_MAP_SWIZZLE_128B
                                : (box[0] * 2 == 64) ? CU_TENSOR_MAP_SWIZZLE_64B
                                                     : CU_TENSOR_MAP_SWIZZLE_32B;
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(RC_ERR_CUDA, "%s: cuTensorMapEncodeTiled failed (%d)", what, (int)r);
  return RC_OK;
}

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
// sgn(x[h][w] - x[h+1][w]), each a 2-bit two's-complement -1 / 0 / +1 (0 past the last column / row) -- which is all the
// smoothness BACKWARD needs (rc_tv_bwd_codes: 0.5 bytes per element read instead of x again).
#ifndef RC_PREPASS_TV_UNROLL
#define RC_PREPASS_TV_UNROLL 1
#endif
#ifndef RC_PREPASS_TV_THREADS
#define RC_PREPASS_TV_THREADS 128
#endif
#ifndef RC_PREPASS_TV_BLOCKS
#define RC_PREPASS_TV_BLOCKS 4
#endif
constexpr int kPrepassTvUnroll = RC_PREPASS_TV_UNROLL;
constexpr int kPrepassTvThreads = RC_PREPASS_TV_THREADS;
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
__global__ void __launch_bounds__(kPrepassTvThreads, RC_PREPASS_TV_BLOCKS)
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

// ------------------------------------------------------------------------------------------------
// main kernel
// ------------------------------------------------------------------------------------------------
constexpr int kTilePx = 128;
constexpr int kThreads = 384;          // 12 warps: 0 TMA, 1 MMA, 2 TMEM alloc, 3 spare, 4-11 compute (softmax, then dX epilogue)
constexpr int kStages = 4;             // ring of 32 KB slots, each with its own full/empty barrier
constexpr int kStageBytes = 32 * 1024; // one slot = two X chunks (2 x 16 KB) | one text chunk (<= 32 KB) | T^T [128 d][<=128 k]
constexpr int kPBytes = 64 * 1024;     // P [128 px][<=256 k] bf16, four K-major 128B-swizzled sub-tiles
constexpr int kStgBufs = 3;             // dX staging buffers; X for the epilogue is prefetched kStgBufs-1 steps ahead
constexpr int kStgPx = 32;             // pixels per dX staging step
constexpr int kStgBytes = 128 * kStgPx * 2;   // [128 d][32 px] bf16 = 8 KB
constexpr int kTmemCols = 512;
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

struct __align__(8) UmmaBars {
  uint64_t full[kStages], empty[kStages];
  uint64_t s_full, s_empty, p_full, p_empty;
  uint64_t acc_full[2], acc_empty[2];
  uint64_t stg_full[kStgBufs], stg_done[kStgBufs];
  uint32_t tmem_base;
  uint32_t pad;
};

constexpr int kOffP = kStages * kStageBytes;
constexpr int kOffStg = kOffP + kPBytes;
constexpr int kScaleBufs = 4;          // per-tile row-scale buffers (softmax runs up to 2 tiles ahead of the dX epilogue)
constexpr int kOffScale = kOffStg + kStgBufs * kStgBytes;       // rs[4][128], cs[4][128] floats
constexpr int kOffXch = kOffScale + 2 * kScaleBufs * 128 * 4;   // softmax half<->half exchange: max, sum, sez, sy [2][128] each
constexpr int kOffBars = kOffXch + 4 * 2 * 128 * 4;
constexpr int kSmemBytes = kOffBars + (int)sizeof(UmmaBars) + 1024;   // + alignment slack

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// mbar_wait that also accumulates the cycles spent waiting (per role, reported for CTA 0)
#ifdef RC_TIMING
#define RC_T0(name) const long long name = clock64()
#define RC_TACC(idx, name) wt[idx] += clock64() - name
__device__ __forceinline__ void mbar_wait_t(uint64_t* bar, uint32_t parity, int tag, long long* acc) {
  const long long t0 = clock64();
  mbar_wait(bar, parity, tag);
  acc[tag] += clock64() - t0;
}
#else
#define RC_T0(name)
#define RC_TACC(idx, name)
__device__ __forceinline__ void mbar_wait_t(uint64_t* bar, uint32_t parity, int tag, long long*) {
  mbar_wait(bar, parity, tag);
}
#endif

struct InfoNceParams {
  int B, D, K, Kp;
  int64_t HW;
  int tiles_per_img;
  int n_tiles;
  const float* inv_norm;
  const int32_t* y;
  const float* w;
  float inv_tau;
  const float* grad_scale;
  const double* w_sum_in;
  float* lse;
  double* loss_sum;
  double* w_sum;
  double* dlogtau;
  long long* dbg;   // optional [32] per-tag wait-cycle counters of CTA 0 (bring-up instrumentation)
};

template <bool kBwd>
__global__ void __launch_bounds__(kThreads, 1)
infonce_umma_kernel(const __grid_constant__ CUtensorMap map_x_s,   // X [B][D][HW], box (64 px, 64 d, 1)
                    const __grid_constant__ CUtensorMap map_t,     // T [Kp][D],    box (64 d, Kp)
                    const __grid_constant__ CUtensorMap map_tt,    // T^T [D][Kp],  box (64 k, 128 d)
                    const __grid_constant__ CUtensorMap map_x_e,   // X,            box (32 px, 128 d, 1)
                    const __grid_constant__ CUtensorMap map_dx,    // dX,           box (32 px, 128 d, 1)
                    const InfoNceParams prm) {
  // 1024-byte alignment (128B-swizzle atoms) comes from the declaration, so that the compiler keeps the
  // shared address space (LDS/STS instead of generic LD/ST) for every access derived from `smem`.
  extern __shared__ __align__(1024) uint8_t smem[];
  UmmaBars* bars = reinterpret_cast<UmmaBars*>(smem + kOffBars);
  float* rs_s = reinterpret_cast<float*>(smem + kOffScale);          // [kScaleBufs][128]
  float* cs_s = rs_s + kScaleBufs * 128;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_dchunks = prm.D / 64;
  const int n_q = prm.D / 128;
  const int n_kchunks = prm.Kp / 64;
  const int n_units = (n_kchunks + 1) / 2;   // dX phase pipeline units (<= 2 k-chunks each) per channel block

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_x_s); tma_prefetch_desc(&map_t);
    if (kBwd) { tma_prefetch_desc(&map_tt); tma_prefetch_desc(&map_x_e); tma_prefetch_desc(&map_dx); }
    for (int i = 0; i < kStages; ++i) { mbar_init(&bars->full[i], 1); mbar_init(&bars->empty[i], 1); }
    mbar_init(&bars->s_full, 1); mbar_init(&bars->s_empty, 256);
    mbar_init(&bars->p_full, 256); mbar_init(&bars->p_empty, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&bars->acc_full[i], 1); mbar_init(&bars->acc_empty[i], 256); }
    for (int i = 0; i < kStgBufs; ++i) { mbar_init(&bars->stg_full[i], 1); mbar_init(&bars->stg_done[i], 256); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<kTmemCols>(&bars->tmem_base);
  if (kBwd) {
    for (int i = threadIdx.x; i < kPBytes / 16; i += kThreads) reinterpret_cast<uint4*>(smem + kOffP)[i] = make_uint4(0, 0, 0, 0);
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = bars->tmem_base;
#ifdef RC_TIMING
  long long wt[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) wt[i] = 0;
  const long long t_start = clock64();
#else
  long long* wt = nullptr;
#endif
  const uint32_t idesc_s = make_idesc_bf16(128, prm.Kp, /*A MN-major*/ 1, /*B K-major*/ 0);
  const uint32_t idesc_d = make_idesc_bf16(128, 128, 0, 0);

  if (warp == 0 && lane == 0) {
    // =============================== TMA producer ===============================
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < prm.n_tiles; tile += gridDim.x) {
      const int b = tile / prm.tiles_per_img;
      const int px0 = (tile - b * prm.tiles_per_img) * kTilePx;
      for (int cp = 0; cp < n_dchunks / 2; ++cp) {
        {   // slot A: X chunks 2cp, 2cp+1 -- [64 d][128 px] each, as two 64-pixel boxes
          const int st = it % kStages;
          mbar_wait_t(&bars->empty[st], ((it / kStages) & 1) ^ 1, 1, wt);
          uint8_t* sb = smem + st * kStageBytes;
          mbar_arrive_expect_tx(&bars->full[st], 4 * 8192);
          for (int cc = 0; cc < 2; ++cc) {
            tma_load_3d(sb + cc * 16384, &map_x_s, &bars->full[st], px0, (2 * cp + cc) * 64, b);
            tma_load_3d(sb + cc * 16384 + 8192, &map_x_s, &bars->full[st], px0 + 64, (2 * cp + cc) * 64, b);
          }
          ++it;
        }
        for (int cc = 0; cc < 2; ++cc, ++it) {   // slots B, C: text chunks [Kp][64 d]
          const int st = it % kStages;
          mbar_wait_t(&bars->empty[st], ((it / kStages) & 1) ^ 1, 1, wt);
          mbar_arrive_expect_tx(&bars->full[st], prm.Kp * 128);
          tma_load_2d(smem + st * kStageBytes, &map_t, &bars->full[st], (2 * cp + cc) * 64, 0);
        }
      }
      if (kBwd) {
        for (int q = 0; q < n_q; ++q)
          for (int u = 0; u < n_units; ++u, ++it) {
            const int st = it % kStages;
            mbar_wait_t(&bars->empty[st], ((it / kStages) & 1) ^ 1, 2, wt);
            uint8_t* sb = smem + st * kStageBytes;
            const int nb = min(2, n_kchunks - 2 * u);
            mbar_arrive_expect_tx(&bars->full[st], nb * 16384);
            for (int jj = 0; jj < nb; ++jj)
              tma_load_2d(sb + jj * 16384, &map_tt, &bars->full[st], (2 * u + jj) * 64, q * 128);
          }
      }
    }
  } else if (warp == 1 && lane == 0) {
    // =============================== MMA issuer ================================
    uint32_t it = 0, lt = 0, qcount = 0;
    for (int tile = blockIdx.x; tile < prm.n_tiles; tile += gridDim.x, ++lt) {
      mbar_wait_t(&bars->s_empty, (lt & 1) ^ 1, 3, wt);
      tc_fence_after();
      for (int cp = 0; cp < n_dchunks / 2; ++cp, it += 3) {
        const int sa = it % kStages;
        mbar_wait_t(&bars->full[sa], (it / kStages) & 1, 4, wt);
        const uint32_t xa = smem_u32(smem + sa * kStageBytes);
        for (int cc = 0; cc < 2; ++cc) {
          const uint32_t jt = it + 1 + cc;
          const int sbt = jt % kStages;
          mbar_wait_t(&bars->full[sbt], (jt / kStages) & 1, 4, wt);
          tc_fence_after();
          const uint32_t tb = smem_u32(smem + sbt * kStageBytes);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            // A: X chunk [64 d][128 px], MN-major; one k-step = 16 channels = two 1024-byte atoms
            const uint64_t a = desc_mnmajor_sw128(xa + cc * 16384 + ks * 2048, 8192);
            const uint64_t bdesc = desc_kmajor_sw128(tb + ks * 32);
            mma_bf16_ss(tmem, a, bdesc, idesc_s, (cp | cc | ks) != 0);
          }
          mma_commit(&bars->empty[sbt]);
        }
        mma_commit(&bars->empty[sa]);
      }
      mma_commit(&bars->s_full);
      if (kBwd) {
        mbar_wait_t(&bars->p_full, lt & 1, 5, wt);
        tc_fence_after();
        const uint32_t pb = smem_u32(smem + kOffP);
        for (int q = 0; q < n_q; ++q, ++qcount) {
          const int ab = qcount & 1;
          mbar_wait_t(&bars->acc_empty[ab], ((qcount >> 1) & 1) ^ 1, 6, wt);
          tc_fence_after();
          const uint32_t dcol = tmem + 256 + ab * 128;
          for (int u = 0; u < n_units; ++u, ++it) {
            const int st = it % kStages;
            mbar_wait_t(&bars->full[st], (it / kStages) & 1, 7, wt);
            tc_fence_after();
            const uint32_t sb = smem_u32(smem + st * kStageBytes);
            const int nb = min(2, n_kchunks - 2 * u);
            for (int jj = 0; jj < nb; ++jj) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                const uint64_t a = desc_kmajor_sw128(sb + jj * 16384 + ks * 32);             // T^T [128 d][64 k]
                const uint64_t bdesc = desc_kmajor_sw128(pb + (2 * u + jj) * 16384 + ks * 32);   // P [128 px][64 k]
                mma_bf16_ss(dcol, a, bdesc, idesc_d, (u | jj | ks) != 0);
              }
            }
            mma_commit(&bars->empty[st]);
          }
          mma_commit(&bars->acc_full[ab]);
        }
        mma_commit(&bars->p_empty);
      }
    }
  } else if (kBwd && warp == 3 && lane == 0) {
    // ================= staging DMA: TMA loads of X for the dX epilogue, TMA stores of dX =================
    const int steps_per_tile = n_q * 4;
    const int64_t my_tiles = (prm.n_tiles > (int)blockIdx.x) ? (prm.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const int64_t total_steps = my_tiles * steps_per_tile;
    struct Cursor { int tile, rem, buf, b, px0; };
    auto init = [&](Cursor& c) {
      c.tile = blockIdx.x; c.rem = 0; c.buf = 0;
      c.b = c.tile / prm.tiles_per_img; c.px0 = (c.tile - c.b * prm.tiles_per_img) * kTilePx;
    };
    auto advance = [&](Cursor& c) {
      c.buf = (c.buf + 1 == kStgBufs) ? 0 : c.buf + 1;
      if (++c.rem == steps_per_tile) {
        c.rem = 0; c.tile += gridDim.x;
        c.b = c.tile / prm.tiles_per_img; c.px0 = (c.tile - c.b * prm.tiles_per_img) * kTilePx;
      }
    };
    Cursor ld, stc;
    init(ld); init(stc);
    auto issue_next_load = [&]() {
      mbar_arrive_expect_tx(&bars->stg_full[ld.buf], kStgBytes);
      tma_load_3d(smem + kOffStg + ld.buf * kStgBytes, &map_x_e, &bars->stg_full[ld.buf], ld.px0 + (ld.rem & 3) * kStgPx,
                  (ld.rem >> 2) * 128, ld.b);
      advance(ld);
    };
    for (int i = 0; i < kStgBufs - 1; ++i)
      if (i < total_steps) issue_next_load();
    uint32_t par = 0;
    for (int64_t s = 0; s < total_steps; ++s) {
      mbar_wait_t(&bars->stg_done[stc.buf], par, 13, wt);
      tma_store_3d(&map_dx, smem + kOffStg + stc.buf * kStgBytes, stc.px0 + (stc.rem & 3) * kStgPx, (stc.rem >> 2) * 128, stc.b);
      tma_store_commit();
      if (stc.buf + 1 == kStgBufs) par ^= 1;
      advance(stc);
      if (s + kStgBufs - 1 < total_steps) {
        tma_store_wait_read0_keep1();     // the store of step s-1 has finished reading the buffer being refilled
        issue_next_load();
      }
    }
    tma_store_wait_all0();
  } else if (warp >= 4) {
    // ============ compute warps: softmax / CE of the tile, then its dX epilogue ============
    // Two warps per TMEM lane quarter: half 0 (warps 4-7) owns text columns [0, Kp/2) in the softmax and pixels
    // [0,16) of every 32-pixel staging step in the epilogue; half 1 (warps 8-11) the rest.
    const int half = warp >= 8 ? 1 : 0;
    const int row = (warp & 3) * 32 + lane;                 // pixel within the tile == TMEM lane
    const int Kh = prm.Kp >> 1;                             // columns per half (multiple of 32)
    const int cb = half * Kh;
    const uint32_t trow = tmem + ((uint32_t)((warp & 3) * 32) << 16) + cb;
    uint8_t* prow = smem + kOffP + row * 128;
    const int sw = row & 7;
    float* xch = reinterpret_cast<float*>(smem + kOffXch);  // [4][2][128]
    float loss_acc = 0.f, w_acc = 0.f, dlt_acc = 0.f;
    float inv_wsum = 0.f;
    float gscale = 1.f;
    if (kBwd) {
      const double ws = prm.w_sum_in[0];
      inv_wsum = ws > 0.0 ? (float)(1.0 / ws) : 0.f;
      if (prm.grad_scale) gscale = prm.grad_scale[0];
    }
    // epilogue state
    const uint32_t trow_acc = tmem + ((uint32_t)((warp & 3) * 32) << 16) + 256 + half * 16;
    int sb = 0;
    uint32_t sb_par = 0, qcount = 0;
    float nx_inv_n = 0.f, nx_w = 0.f;
    int nx_y = -1;
    auto load_pixel_scalars = [&](int t) {
      nx_inv_n = 0.f; nx_w = 0.f; nx_y = -1;
      if (t < prm.n_tiles) {
        const int tb = t / prm.tiles_per_img;
        const int tpx = (t - tb * prm.tiles_per_img) * kTilePx + row;
        if (tpx < prm.HW) {
          const int64_t tm = (int64_t)tb * prm.HW + tpx;
          nx_inv_n = __ldg(prm.inv_norm + tm);
          nx_y = __ldg(prm.y + tm);
          nx_w = __ldg(prm.w + tm);
        }
      }
    };
    load_pixel_scalars(blockIdx.x);
    // exp(z - m) needs m >= max z for range only.  Cosine logits are bounded: |z| <= |t_k| / tau, so for
    // tau not too small the constant m = 1.01 / tau replaces the row-maximum pass over TMEM.
    const bool use_bound = prm.inv_tau * (2.02f * kLog2e) < 100.f;
    const float ml_bound = prm.inv_tau * (1.01f * kLog2e);
    uint32_t lt = 0;
    for (int tile = blockIdx.x; tile < prm.n_tiles; tile += gridDim.x, ++lt) {
      RC_T0(tg0);
      const int b = tile / prm.tiles_per_img;
      const int px = (tile - b * prm.tiles_per_img) * kTilePx + row;
      const bool valid = px < prm.HW;
      const int64_t m = (int64_t)b * prm.HW + px;
      const float inv_n = nx_inv_n;
      const int yi = nx_y;
      const float wi = yi >= 0 ? nx_w : 0.f;
      load_pixel_scalars(tile + (int)gridDim.x);          // next tile's scalars: latency hidden behind this tile
      const float zs = inv_n * prm.inv_tau;     // z = s * zs   (zs >= 0)
      const float zl = zs * kLog2e;
      RC_TACC(5, tg0);
      mbar_wait_t(&bars->s_full, lt & 1, 8, wt);
      tc_fence_after();
      RC_T0(tp1);
      // pass 1: maximum of the raw dots over this half's valid columns (skipped when the bound applies)
      float mx = -FLT_MAX;
      for (int c = 0; !use_bound && c * 32 < Kh; ++c) {
        const int nvalid = prm.K - (cb + c * 32);
        if (nvalid <= 0) break;
        uint32_t r[32];
        tmem_ld_32x32(trow + c * 32, r);
        tmem_ld_wait();
        float m0 = -FLT_MAX, m1 = -FLT_MAX, m2 = -FLT_MAX, m3 = -FLT_MAX;
        if (nvalid >= 32) {
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            m0 = fmaxf(m0, __uint_as_float(r[i])); m1 = fmaxf(m1, __uint_as_float(r[i + 1]));
            m2 = fmaxf(m2, __uint_as_float(r[i + 2])); m3 = fmaxf(m3, __uint_as_float(r[i + 3]));
          }
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) if (i < nvalid) m0 = fmaxf(m0, __uint_as_float(r[i]));
        }
        mx = fmaxf(fmaxf(mx, fmaxf(m0, m1)), fmaxf(m2, m3));
      }
      float ml = ml_bound;
      if (!use_bound) {
        xch[(0 * 2 + half) * 128 + row] = mx;
        named_bar_sync(2, 256);
        mx = fmaxf(mx, xch[(0 * 2 + (half ^ 1)) * 128 + row]);
        ml = mx * zl;
      }
      RC_TACC(6, tp1);
      if (kBwd) mbar_wait_t(&bars->p_empty, (lt & 1) ^ 1, 9, wt);
      RC_T0(tp2);
      // pass 2: e = exp(z - m), partial sums, P (bf16, K-major 128B-swizzled sub-tiles)
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f, q0 = 0.f, q1 = 0.f, q2 = 0.f, q3 = 0.f, sy = 0.f;
      for (int c = 0; c * 32 < Kh; ++c) {
        const int k0 = cb + c * 32;
        const int nvalid = prm.K - k0;
        if (nvalid <= 0) break;
        uint32_t r[32];
        tmem_ld_32x32(trow + c * 32, r);
        tmem_ld_wait();
        const int yrel = yi - k0;
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          const float a0 = __uint_as_float(r[i]), a1 = __uint_as_float(r[i + 1]);
          const float a2 = __uint_as_float(r[i + 2]), a3 = __uint_as_float(r[i + 3]);
          float e0 = fast_exp2(fminf(fmaf(a0, zl, -ml), 64.f)), e1 = fast_exp2(fminf(fmaf(a1, zl, -ml), 64.f));
          float e2 = fast_exp2(fminf(fmaf(a2, zl, -ml), 64.f)), e3 = fast_exp2(fminf(fmaf(a3, zl, -ml), 64.f));
          if (nvalid < 32) {      // warp-uniform; only the chunk that straddles K
            e0 = (i < nvalid) ? e0 : 0.f; e1 = (i + 1 < nvalid) ? e1 : 0.f;
            e2 = (i + 2 < nvalid) ? e2 : 0.f; e3 = (i + 3 < nvalid) ? e3 : 0.f;
          }
          s0 += e0; s1 += e1; s2 += e2; s3 += e3;
          q0 = fmaf(e0, a0, q0); q1 = fmaf(e1, a1, q1); q2 = fmaf(e2, a2, q2); q3 = fmaf(e3, a3, q3);
          sy = (yrel == i) ? a0 : sy; sy = (yrel == i + 1) ? a1 : sy;
          sy = (yrel == i + 2) ? a2 : sy; sy = (yrel == i + 3) ? a3 : sy;
          pk[i >> 1] = pack_bf16x2(e0, e1);
          pk[(i >> 1) + 1] = pack_bf16x2(e2, e3);
        }
        if (kBwd) {
          uint8_t* sub = prow + (k0 >> 6) * 16384;          // 64-wide K sub-tile
          const int cbase = (k0 & 32) >> 3;                 // first 16-byte chunk of this 32-column group
#pragma unroll
          for (int g = 0; g < 4; ++g)
            *reinterpret_cast<uint4*>(sub + (((cbase + g) ^ sw) << 4)) = make_uint4(pk[g * 4], pk[g * 4 + 1], pk[g * 4 + 2], pk[g * 4 + 3]);
        }
      }
      tc_fence_before();
      mbar_arrive(&bars->s_empty);               // S columns may be overwritten by the next tile
      RC_TACC(7, tp2);
      RC_T0(tp3);
      float sum = (s0 + s1) + (s2 + s3);
      float sez = (q0 + q1) + (q2 + q3);
      const bool mine_y = yi >= cb && yi < cb + Kh;
      xch[(1 * 2 + half) * 128 + row] = sum;
      xch[(2 * 2 + half) * 128 + row] = sez;
      xch[(3 * 2 + half) * 128 + row] = mine_y ? sy : 0.f;
      named_bar_sync(2, 256);
      sum += xch[(1 * 2 + (half ^ 1)) * 128 + row];
      sez += xch[(2 * 2 + (half ^ 1)) * 128 + row];
      sy = mine_y ? sy : xch[(3 * 2 + (half ^ 1)) * 128 + row];
      const float zy = sy * zs;
      if (half == 0) {
        const float lse = (ml + __log2f(sum)) * kLn2;
        loss_acc += wi * (lse - zy);
        w_acc += wi;
        if (valid && prm.lse) prm.lse[m] = lse;
      }
      if (kBwd) {
        const float coef = gscale * wi * inv_wsum;
        const float inv_sum = 1.f / sum;
        if (mine_y) {    // P[row][y] = e_y - sum  (softmax - onehot, times sum), subtraction before rounding
          const float ey = fast_exp2(fminf(fmaf(sy, zl, -ml), 64.f));
          const int kk = yi & 63;
          uint8_t* sub = prow + (yi >> 6) * 16384;
          *reinterpret_cast<__nv_bfloat16*>(sub + (((kk >> 3) ^ sw) << 4) + (kk & 7) * 2) = __float2bfloat16_rn(ey - sum);
        }
        if (half == 0) {
          const float cj = coef * (sez * zs * inv_sum - zy);        // sum_k dz_k z_k
          rs_s[(lt & (kScaleBufs - 1)) * 128 + row] = inv_n * prm.inv_tau * coef * inv_sum;
          cs_s[(lt & (kScaleBufs - 1)) * 128 + row] = inv_n * inv_n * cj;
          dlt_acc -= cj;
        }
        fence_proxy_async_smem();                 // P is read by the tensor core (async proxy)
        mbar_arrive(&bars->p_full);
        named_bar_sync(2, 256);                   // rs/cs written by half 0 are visible to all compute warps
      }
      RC_TACC(10, tp3);
      if (!kBwd) continue;
      // ------------------------------ dX epilogue of this tile ------------------------------
      const int px0 = (tile - b * prm.tiles_per_img) * kTilePx;
      const float* rs = rs_s + (lt & (kScaleBufs - 1)) * 128;
      const float* cs = cs_s + (lt & (kScaleBufs - 1)) * 128;
      for (int q = 0; q < n_q; ++q, ++qcount) {
        const int ab = qcount & 1;
        mbar_wait_t(&bars->acc_full[ab], (qcount >> 1) & 1, 11, wt);
        tc_fence_after();
        for (int h = 0; h < 4; ++h) {
          // this thread: channel row `row`, pixels [h*32 + half*16, +16) of the tile
          uint32_t acc[16];
          RC_T0(tl0);
          tmem_ld_32x16(trow_acc + ab * 128 + h * kStgPx, acc);
          tmem_ld_wait();
          RC_TACC(15, tl0);
          if (h == 3) { tc_fence_before(); mbar_arrive(&bars->acc_empty[ab]); }
          mbar_wait_t(&bars->stg_full[sb], sb_par, 12, wt);
          RC_T0(tc0);
          uint8_t* srow = smem + kOffStg + sb * kStgBytes + row * 64;    // 32 px bf16 = 64 B per channel row
          const int sw64 = (row >> 1) & 3;                                // 64-byte swizzle
          const float* rsp = rs + h * kStgPx + half * 16;
          const float* csp = cs + h * kStgPx + half * 16;
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            uint4* p = reinterpret_cast<uint4*>(srow + (((half * 2 + g) ^ sw64) << 4));
            const uint4 xv = *p;
            const uint32_t xu[4] = {xv.x, xv.y, xv.z, xv.w};
            const float4 r0 = *reinterpret_cast<const float4*>(rsp + g * 8);
            const float4 r1 = *reinterpret_cast<const float4*>(rsp + g * 8 + 4);
            const float4 c0 = *reinterpret_cast<const float4*>(csp + g * 8);
            const float4 c1 = *reinterpret_cast<const float4*>(csp + g * 8 + 4);
            const float rr[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
            const float cc[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
            float o[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float xval = (i & 1) ? __uint_as_float(xu[i >> 1] & 0xffff0000u) : __uint_as_float(xu[i >> 1] << 16);
              o[i] = fmaf(rr[i], __uint_as_float(acc[g * 8 + i]), -cc[i] * xval);
            }
            uint4 ov;
            ov.x = pack_bf16x2(o[0], o[1]); ov.y = pack_bf16x2(o[2], o[3]);
            ov.z = pack_bf16x2(o[4], o[5]); ov.w = pack_bf16x2(o[6], o[7]);
            *p = ov;
          }
          RC_TACC(1, tc0);
          fence_proxy_async_smem();                 // staged dX is read by the TMA store (async proxy)
          mbar_arrive(&bars->stg_done[sb]);         // the DMA thread stores this buffer and refills it
          if (++sb == kStgBufs) { sb = 0; sb_par ^= 1; }
        }
      }
    }
    if (half == 0) {
      loss_acc = warp_sum(loss_acc); w_acc = warp_sum(w_acc); dlt_acc = warp_sum(dlt_acc);
      if (lane == 0) {
        if (prm.loss_sum) atomicAdd(prm.loss_sum, (double)loss_acc);
        if (prm.w_sum) atomicAdd(prm.w_sum, (double)w_acc);
        if (kBwd && prm.dlogtau) atomicAdd(prm.dlogtau, (double)dlt_acc);
      }
    }
  }
#ifdef RC_TIMING
  if (prm.dbg != nullptr && blockIdx.x == 0 && lane == 0 && (warp == 0 || warp == 1 || warp == 4)) {
    wt[0] = clock64() - t_start;
    const int role = warp == 0 ? 0 : (warp == 1 ? 1 : 2);
#pragma unroll
    for (int i = 0; i < 16; ++i) prm.dbg[role * 16 + i] = wt[i];
  }
#endif
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<kTmemCols>(tmem);
  }
}

}  // namespace rc

// ------------------------------------------------------------------------------------------------
// bring-up kernel: one 128 x N x Kd GEMM tile through the same TMA / descriptor / tcgen05 / TMEM path
// ------------------------------------------------------------------------------------------------
namespace rc {

struct __align__(8) DebugBars { uint64_t full, done; uint32_t tmem_base, pad; };

__global__ void __launch_bounds__(128, 1)
debug_umma_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, int N, int Kd,
                       int variant, float* __restrict__ c) {
  // 1024-byte alignment (128B-swizzle atoms) comes from the declaration, so that the compiler keeps the
  // shared address space (LDS/STS instead of generic LD/ST) for every access derived from `smem`.
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sa = smem;               // 16 KB
  uint8_t* sbm = smem + 16384;      // <= 32 KB
  DebugBars* bars = reinterpret_cast<DebugBars*>(smem + 49152);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    mbar_init(&bars->full, 1);
    mbar_init(&bars->done, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<256>(&bars->tmem_base);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = bars->tmem_base;
  if (threadIdx.x == 0) {
    const uint32_t idesc = make_idesc_bf16(128, N, variant == 0 ? 0 : 1, 0);
    for (int ck = 0; ck < Kd / 64; ++ck) {
      mbar_arrive_expect_tx(&bars->full, 16384 + N * 128);
      if (variant == 0) {
        tma_load_2d(sa, &map_a, &bars->full, ck * 64, 0);             // A [128][Kd]: box (64 k, 128 rows)
      } else {
        tma_load_2d(sa, &map_a, &bars->full, 0, ck * 64);             // A^T [Kd][128]: box (64 m, 64 k) x 2
        tma_load_2d(sa + 8192, &map_a, &bars->full, 64, ck * 64);
      }
      tma_load_2d(sbm, &map_b, &bars->full, ck * 64, 0);              // B [N][Kd]: box (64 k, N rows)
      mbar_wait(&bars->full, ck & 1, 100);
      tc_fence_after();
      for (int ks = 0; ks < 4; ++ks) {
        uint64_t a;
        if (variant == 0) a = desc_kmajor_sw128(smem_u32(sa) + ks * 32);
        else if (variant == 1) a = desc_mnmajor_sw128(smem_u32(sa) + ks * 2048, 8192);
        else a = make_smem_desc_sw128(smem_u32(sa) + ks * 2048, 1024, 8192);   // hypothesis: LBO/SBO roles swapped
        const uint64_t b = desc_kmajor_sw128(smem_u32(sbm) + ks * 32);
        mma_bf16_ss(tmem, a, b, idesc, (ck | ks) != 0);
      }
      mma_commit(&bars->done);
      mbar_wait(&bars->done, ck & 1, 101);
    }
  }
  __syncthreads();
  tc_fence_after();
  const int row = warp * 32 + lane;
  for (int cc = 0; cc < N / 32; ++cc) {
    uint32_t r[32];
    tmem_ld_32x32(tmem + ((uint32_t)(warp * 32) << 16) + cc * 32, r);
    tmem_ld_wait();
    for (int i = 0; i < 32; ++i) c[(int64_t)row * N + cc * 32 + i] = __uint_as_float(r[i]);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) { tc_fence_after(); tmem_dealloc<256>(tmem); }
}

static int check_sm100(const char* what) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return fail(RC_ERR_NO_DEVICE, "%s: no CUDA device", what);
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (major != 10) return fail(RC_ERR_NO_DEVICE, "%s: needs an sm_100 device (compute capability %d.x found)", what, major);
  return RC_OK;
}

}  // namespace rc

#ifdef RC_BRINGUP
extern "C" int rc_debug_umma_gemm(const void* a_bf16, const void* b_bf16, int N, int Kd, int variant, float* c, void* stream) {
  RC_REQUIRE(a_bf16 && b_bf16 && c, "rc_debug_umma_gemm: null pointer");
  RC_REQUIRE(N >= 32 && N <= 256 && N % 32 == 0 && Kd >= 64 && Kd % 64 == 0 && variant >= 0 && variant <= 2,
             "rc_debug_umma_gemm: bad shape N=%d Kd=%d variant=%d", N, Kd, variant);
  int rcode = rc::check_sm100("rc_debug_umma_gemm");
  if (rcode) return rcode;
  CUtensorMap ma, mb;
  if (variant == 0) {
    const uint64_t dims[2] = {(uint64_t)Kd, 128}, str[2] = {2, (uint64_t)Kd * 2};
    const uint32_t box[2] = {64, 128};
    if ((rcode = rc::make_tmap_bf16(&ma, a_bf16, 2, dims, str, box, "debug A"))) return rcode;
  } else {
    const uint64_t dims[2] = {128, (uint64_t)Kd}, str[2] = {2, 256};
    const uint32_t box[2] = {64, 64};
    if ((rcode = rc::make_tmap_bf16(&ma, a_bf16, 2, dims, str, box, "debug A^T"))) return rcode;
  }
  {
    const uint64_t dims[2] = {(uint64_t)Kd, (uint64_t)N}, str[2] = {2, (uint64_t)Kd * 2};
    const uint32_t box[2] = {64, (uint32_t)N};
    if ((rcode = rc::make_tmap_bf16(&mb, b_bf16, 2, dims, str, box, "debug B"))) return rcode;
  }
  const int smem = 49152 + 64 + 1024;
  cudaError_t e = cudaFuncSetAttribute(rc::debug_umma_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return rc::fail(RC_ERR_CUDA, "rc_debug_umma_gemm: smem opt-in: %s", cudaGetErrorString(e));
  rc::debug_umma_gemm_kernel<<<1, 128, smem, (cudaStream_t)stream>>>(ma, mb, N, Kd, variant, c);
  return rc::check_launch("rc_debug_umma_gemm");
}
#endif  // RC_BRINGUP

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

#ifndef RC_PREPASS_TV_ROWS
#define RC_PREPASS_TV_ROWS 4
#endif
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
  constexpr int R = RC_PREPASS_TV_ROWS;
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
                             void* stream, const int32_t* k_dev = nullptr, const float* log_tau_dev = nullptr) {
  using namespace rc;
  RC_REQUIRE(x && t_bf16 && y && w && workspace, "rc_infonce_bf16: null pointer");
  RC_REQUIRE(B >= 0 && HW >= 0, "rc_infonce_bf16: bad shape");
  if (K < 1 || K > 256) return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16: K=%d outside [1,256] (use rc_infonce_f32)", K);
  if (D < 128 || D > 512 || D % 128 != 0) return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16: D=%d must be 128, 256, 384 or 512", D);
  RC_REQUIRE((reinterpret_cast<uintptr_t>(t_bf16) & 15) == 0, "rc_infonce_bf16: t must be 16-byte aligned");
  const bool bwd = dx != nullptr;
  if (bwd) RC_REQUIRE(tt_bf16 && w_sum_in && (reinterpret_cast<uintptr_t>(dx) & 15) == 0, "rc_infonce_bf16: backward needs tt_bf16, w_sum_in and aligned dx");
  if (dlogtau && !bwd) return fail(RC_ERR_INVALID, "rc_infonce_bf16: dlogtau needs dx");
  if (B == 0 || HW == 0) return RC_OK;
  int rcode = check_sm100("rc_infonce_bf16");
  if (rcode) return rcode;
  if ((k_dev != nullptr || log_tau_dev != nullptr) && !infonce_pair_supported(D))
    return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16_dyn: device-side K / log tau need D = 256 or 512 (CTA-pair kernel)");
  cudaStream_t s = (cudaStream_t)stream;
  float* inv_norm; __nv_bfloat16* xb;
  // CTA-pair kernel (cta_group::2) when the channel count allows it; RANGECLIP_B200_INFONCE=1cta forces the
  // single-CTA kernel (kept for D = 128 / 384 and as the A/B baseline).  The pair kernel computes 1/|x_p| itself
  // from the operand tiles in shared memory, so a bf16 input needs no pre-pass at all (an fp32 input still needs
  // its bf16 copy).
#ifdef RC_BRINGUP
  const char* impl = getenv("RANGECLIP_B200_INFONCE");     // bring-up A/B switch; never compiled into the shipped library
#else
  const char* impl = nullptr;
#endif
  const bool use_pair = (rep != 1 || !(impl != nullptr && impl[0] == '1')) && infonce_pair_supported(D);
  const int keep_w = (flags & RC_INFONCE_KEEP_WEIGHT) ? 1 : 0;
  const int acc_dx = (flags & RC_INFONCE_ACCUMULATE_DX) ? 1 : 0;
  const float* lse_in = (flags & RC_INFONCE_LSE_GIVEN) ? lse : nullptr;
  if (acc_dx) RC_REQUIRE(bwd, "rc_infonce_bf16: RC_INFONCE_ACCUMULATE_DX needs dx");
  if (keep_w || lse_in || acc_dx) {
    if (!use_pair || rep != 1 || dt != nullptr)
      return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16: the K-blocked flags need D = 256 or 512, one target per row and no dText");
    RC_REQUIRE(!(flags & RC_INFONCE_LSE_GIVEN) || lse != nullptr, "rc_infonce_bf16: RC_INFONCE_LSE_GIVEN needs lse");
  }
  if (rep != 1) {
    if (!use_pair) return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16_rep4: D=%d must be 256 or 512", D);
    RC_REQUIRE((reinterpret_cast<uintptr_t>(y) & 15) == 0 && (reinterpret_cast<uintptr_t>(w) & 15) == 0,
               "rc_infonce_bf16_rep4: y and w must be 16-byte aligned");
  }
  const bool skip_prepass = (flags & RC_INFONCE_PREPASS_DONE) || (use_pair && x_dtype == RC_BF16);
  if ((rcode = infonce_prepass_impl(x, x_dtype, B, D, HW, workspace, workspace_bytes, skip_prepass ? (cudaStream_t)-1 : s,
                                    &inv_norm, &xb))) return rcode;
  const void* xsrc = (x_dtype == RC_F32) ? (const void*)xb : x;
  if (dt != nullptr) {
    // dText: the pair kernel also writes G = rs (P - sum onehot) (bf16 [B][HW][Kp]) into the workspace, then one
    // split-K GEMM over the pixels (infonce_dt_umma.cu) adds G^T X to dt.
    if (!use_pair || !bwd)
      return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16: dText needs dx and D = 256 or 512 (use rc_infonce_f32 otherwise)");
    const int64_t base = rc_infonce_workspace_bytes(B, D, HW, K, x_dtype);
    RC_REQUIRE(workspace_bytes >= rc_infonce_workspace_bytes_dt(B, D, HW, K, x_dtype), "rc_infonce_bf16: workspace too small for dText");
    uint8_t* ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
    void* g = ws + ((base + 255) / 256) * 256;
    if ((rcode = launch_infonce_pair(xsrc, dx, t_bf16, tt_bf16, B, D, HW, K, inv_norm, y, w, inv_tau, grad_scale, w_sum_in, lse,
                                     loss_sum, w_sum, dlogtau, g, rep, 0, nullptr, 0, 0, k_dev, log_tau_dev, s))) return rcode;
    return launch_infonce_dt(g, xsrc, B, D, HW, K, dt, s);
  }
  if (use_pair) {
    // backward launches: the softmax tile as a tensor-memory operand of the dX GEMM (infonce_ts.cu) unless RC_INFONCE_SS_KERNEL
    if (bwd && !(flags & RC_INFONCE_SS_KERNEL) && k_dev == nullptr && log_tau_dev == nullptr)
      return launch_infonce_ts(xsrc, dx, t_bf16, tt_bf16, B, D, HW, K, y, w, inv_tau, grad_scale, w_sum_in, lse, loss_sum, w_sum,
                               dlogtau, rep, keep_w, lse_in, 0, acc_dx, s);
    return launch_infonce_pair(xsrc, dx, t_bf16, tt_bf16, B, D, HW, K, inv_norm, y, w, inv_tau, grad_scale, w_sum_in, lse,
                               loss_sum, w_sum, dlogtau, nullptr, rep, keep_w, lse_in, 0, acc_dx, k_dev, log_tau_dev, s);
  }
  const int Kp = (K + 63) / 64 * 64;
  CUtensorMap m_xs, m_t, m_tt, m_xe, m_dx;
  {
    const uint64_t dims[3] = {(uint64_t)HW, (uint64_t)D, (uint64_t)B};
    const uint64_t str[3] = {2, (uint64_t)HW * 2, (uint64_t)D * HW * 2};
    const uint32_t box_s[3] = {64, 64, 1}, box_e[3] = {kStgPx, 128, 1};
    if ((rcode = make_tmap_bf16(&m_xs, xsrc, 3, dims, str, box_s, "map_x_s"))) return rcode;
    if ((rcode = make_tmap_bf16(&m_xe, xsrc, 3, dims, str, box_e, "map_x_e"))) return rcode;
    if ((rcode = make_tmap_bf16(&m_dx, bwd ? dx : xsrc, 3, dims, str, box_e, "map_dx"))) return rcode;
    const uint64_t tdims[2] = {(uint64_t)D, (uint64_t)Kp}, tstr[2] = {2, (uint64_t)D * 2};
    const uint32_t tbox[2] = {64, (uint32_t)Kp};
    if ((rcode = make_tmap_bf16(&m_t, t_bf16, 2, tdims, tstr, tbox, "map_t"))) return rcode;
    const uint64_t ttdims[2] = {(uint64_t)Kp, (uint64_t)D}, ttstr[2] = {2, (uint64_t)Kp * 2};
    const uint32_t ttbox[2] = {64, 128};
    if ((rcode = make_tmap_bf16(&m_tt, bwd ? tt_bf16 : t_bf16, 2, bwd ? ttdims : tdims, bwd ? ttstr : tstr,
                                bwd ? ttbox : tbox, "map_tt"))) return rcode;
  }
  InfoNceParams prm;
  prm.B = B; prm.D = D; prm.K = K; prm.Kp = Kp; prm.HW = HW;
  prm.tiles_per_img = (int)((HW + kTilePx - 1) / kTilePx);
  if ((int64_t)B * prm.tiles_per_img > 0x7fffffff) return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16: too many tiles");
  prm.n_tiles = B * prm.tiles_per_img;
  prm.inv_norm = inv_norm; prm.y = y; prm.w = w; prm.inv_tau = inv_tau; prm.grad_scale = grad_scale;
  prm.w_sum_in = w_sum_in; prm.lse = lse; prm.loss_sum = loss_sum; prm.w_sum = w_sum; prm.dlogtau = dlogtau; prm.dbg = g_dbg_buf;
  const int grid = prm.n_tiles < num_sms() ? prm.n_tiles : num_sms();
  cudaError_t e;
  if (bwd) {
    e = cudaFuncSetAttribute(infonce_umma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
    if (e != cudaSuccess) return fail(RC_ERR_CUDA, "rc_infonce_bf16: smem opt-in: %s", cudaGetErrorString(e));
    infonce_umma_kernel<true><<<grid, kThreads, kSmemBytes, s>>>(m_xs, m_t, m_tt, m_xe, m_dx, prm);
  } else {
    e = cudaFuncSetAttribute(infonce_umma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
    if (e != cudaSuccess) return fail(RC_ERR_CUDA, "rc_infonce_bf16: smem opt-in: %s", cudaGetErrorString(e));
    infonce_umma_kernel<false><<<grid, kThreads, kSmemBytes, s>>>(m_xs, m_t, m_tt, m_xe, m_dx, prm);
  }
  return check_launch("rc_infonce_bf16");
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

extern "C" int rc_infonce_bf16_kblocks(const void* x, rc_dtype x_dtype, int D, int64_t HW, const void* t_bf16_all,
                                       const void* tt_bf16_all, int K, int n_blocks, const int32_t* y_rel, const float* w_rep,
                                       float inv_tau, float* lse, double* loss_sum, double* w_sum, const double* w_sum_in,
                                       const float* grad_scale, void* dx_blocks, double* dlogtau, void* workspace,
                                       int64_t workspace_bytes, int flags, void* stream) {
  using namespace rc;
  RC_REQUIRE(x && t_bf16_all && y_rel && w_rep && workspace && lse, "rc_infonce_bf16_kblocks: null pointer");
  RC_REQUIRE(HW >= 0 && K >= 1 && n_blocks >= 1 && n_blocks == (K + 255) / 256, "rc_infonce_bf16_kblocks: n_blocks must be ceil(K / 256)");
  if (!infonce_pair_supported(D)) return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16_kblocks: D=%d must be 256 or 512", D);
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
  if (bwd && !(flags & RC_INFONCE_SS_KERNEL))
    return launch_infonce_ts(xsrc, dx_blocks, t_bf16_all, tt_bf16_all, n_blocks, D, HW, K, y_rel, w_rep, inv_tau, grad_scale, w_sum_in,
                             lse, loss_sum, w_sum, dlogtau, 1, 1, lse_in, n_blocks, 0, s);
  return launch_infonce_pair(xsrc, dx_blocks, t_bf16_all, tt_bf16_all, n_blocks, D, HW, K, inv_norm, y_rel, w_rep, inv_tau, grad_scale,
                             w_sum_in, lse, loss_sum, w_sum, dlogtau, nullptr, 1, 1, lse_in, n_blocks, 0, nullptr, nullptr, s);
}

// ------------------------------------------------------------------------------------------------
// bring-up kernel for the CTA-pair (cta_group::2) building blocks: C[256][N] = A[256][Kd] B[N][Kd]^T
// with A rows split 128/128 over the two CTAs and B rows split N/2 / N/2.
// ------------------------------------------------------------------------------------------------
namespace rc {

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128, 1)
debug_umma_gemm_2sm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, int N, int Kd,
                           float* __restrict__ c) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sa = smem;               // 16 KB: own 128 rows of A, one 64-wide K chunk
  uint8_t* sbm = smem + 16384;      // <= 16 KB: own N/2 rows of B
  DebugBars* bars = reinterpret_cast<DebugBars*>(smem + 32768);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  if (threadIdx.x == 0) {
    mbar_init(&bars->full, 1);
    mbar_init(&bars->done, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_2sm<256>(&bars->tmem_base);
  tc_fence_before();
  cluster_sync();
  tc_fence_after();
  const uint32_t tmem = bars->tmem_base;
  if (threadIdx.x == 0) {
    const uint32_t idesc = make_idesc_bf16(256, N, 0, 0);
    const int nh = N / 2;
    for (int ck = 0; ck < Kd / 64; ++ck) {
      if (rank == 0) mbar_arrive_expect_tx(&bars->full, 2 * (16384 + nh * 128));
      tma_load_2d_2sm(sa, &map_a, &bars->full, ck * 64, (int)rank * 128);
      tma_load_2d_2sm(sbm, &map_b, &bars->full, ck * 64, (int)rank * nh);
      if (rank == 0) {
        mbar_wait_cluster(&bars->full, ck & 1, 200);
        tc_fence_after();
        for (int ks = 0; ks < 4; ++ks)
          mma_bf16_ss_2sm(tmem, desc_kmajor_sw128(smem_u32(sa) + ks * 32), desc_kmajor_sw128(smem_u32(sbm) + ks * 32), idesc,
                          (ck | ks) != 0);
        mma_commit_2sm(&bars->done);
      }
      mbar_wait_cluster(&bars->done, ck & 1, 201);   // both CTAs: smem may be refilled, TMEM is current
    }
  }
  __syncthreads();
  tc_fence_after();
  const int row = warp * 32 + lane;
  for (int cc = 0; cc < N / 32; ++cc) {
    uint32_t r[32];
    tmem_ld_32x32(tmem + ((uint32_t)(warp * 32) << 16) + cc * 32, r);
    tmem_ld_wait();
    for (int i = 0; i < 32; ++i) c[((int64_t)rank * 128 + row) * N + cc * 32 + i] = __uint_as_float(r[i]);
  }
  tc_fence_before();
  cluster_sync();
  if (warp == 1) { tc_fence_after(); tmem_dealloc_2sm<256>(tmem); }
}

}  // namespace rc

#ifdef RC_BRINGUP
extern "C" int rc_debug_umma_gemm_2sm(const void* a_bf16, const void* b_bf16, int N, int Kd, float* c, void* stream) {
  RC_REQUIRE(a_bf16 && b_bf16 && c, "rc_debug_umma_gemm_2sm: null pointer");
  RC_REQUIRE(N >= 64 && N <= 256 && N % 64 == 0 && Kd >= 64 && Kd % 64 == 0, "rc_debug_umma_gemm_2sm: bad shape N=%d Kd=%d", N, Kd);
  int rcode = rc::check_sm100("rc_debug_umma_gemm_2sm");
  if (rcode) return rcode;
  CUtensorMap ma, mb;
  {
    const uint64_t dims[2] = {(uint64_t)Kd, 256}, str[2] = {2, (uint64_t)Kd * 2};
    const uint32_t box[2] = {64, 128};
    if ((rcode = rc::make_tmap_bf16(&ma, a_bf16, 2, dims, str, box, "debug2 A"))) return rcode;
    const uint64_t bdims[2] = {(uint64_t)Kd, (uint64_t)N};
    const uint32_t bbox[2] = {64, (uint32_t)(N / 2)};
    if ((rcode = rc::make_tmap_bf16(&mb, b_bf16, 2, bdims, str, bbox, "debug2 B"))) return rcode;
  }
  const int smem = 32768 + 64;
  cudaError_t e = cudaFuncSetAttribute(rc::debug_umma_gemm_2sm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return rc::fail(RC_ERR_CUDA, "rc_debug_umma_gemm_2sm: smem opt-in: %s", cudaGetErrorString(e));
  rc::debug_umma_gemm_2sm_kernel<<<2, 128, smem, (cudaStream_t)stream>>>(ma, mb, N, Kd, c);
  return rc::check_launch("rc_debug_umma_gemm_2sm");
}
#endif  // RC_BRINGUP
