// K5/K6: smoothness (TV-L1) forward sums and backward, shared-memory tiled.
// Replaces RangeCLIP/src/depth_segmentation_model/model.py:332-334 (two F.l1_loss over four
// strided slices) and its autograd (sgn, mul, two slice-scatter adds) with one read of X for the
// forward and one read of X (+ one read-modify-write of dX) for the backward.  sign(0) = 0 as
// torch.sgn (SURVEY Q8: the nearest-upsampled decoder makes half of all differences exactly 0).
#include "common.cuh"

namespace rc {

constexpr int kTvThreads = 256;
constexpr int kTvSmemFloats = 12288 - 64;  // tile budget (rows incl. halo) x W: 48 KB minus the kernels' static shared memory

template <typename T>
__device__ __forceinline__ void tv_load_rows(const T* __restrict__ plane, int H, int W, int h_first, int n_rows,
                                             float* __restrict__ tile, bool vec_ok) {
  // rows h_first .. h_first+n_rows-1 (clamped to the plane; rows outside are left untouched)
  const int lo = h_first < 0 ? 0 : h_first;
  const int hi = (h_first + n_rows) > H ? H : (h_first + n_rows);
  if (hi <= lo) return;
  const T* src = plane + (int64_t)lo * W;
  float* dst = tile + (int64_t)(lo - h_first) * W;
  const int total = (hi - lo) * W;
  if (vec_ok) {
    for (int i = threadIdx.x * 8; i < total; i += kTvThreads * 8) {
      float v[8];
      load8(src + i, v);
#pragma unroll
      for (int j = 0; j < 8; ++j) dst[i + j] = v[j];
    }
  } else {
    for (int i = threadIdx.x; i < total; i += kTvThreads) dst[i] = ElemIO<T>::ld(src + i);
  }
}

template <typename T>
__global__ void __launch_bounds__(kTvThreads)
tv_fwd_kernel(const T* __restrict__ x, int64_t planes, int H, int W, int TH, double* __restrict__ sums) {
  extern __shared__ float tile[];  // [(TH+1)][W]
  const int tiles_per_plane = (H + TH - 1) / TH;
  const int64_t n_tiles = planes * tiles_per_plane;
  const bool vec_ok = (W % 8 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  double acc_h = 0.0, acc_v = 0.0;
  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const int64_t pl = t / tiles_per_plane;
    const int h0 = (int)(t - pl * tiles_per_plane) * TH;
    const int rows = min(TH, H - h0);
    __syncthreads();
    tv_load_rows(x + pl * (int64_t)H * W, H, W, h0, rows + 1, tile, vec_ok);
    __syncthreads();
    const bool has_below = (h0 + rows) < H;
    float sh = 0.f, sv = 0.f;
    for (int i = threadIdx.x; i < rows * W; i += kTvThreads) {
      const int r = i / W, c = i - r * W;
      const float a = tile[i];
      if (c + 1 < W) sh += fabsf(a - tile[i + 1]);
      if (r + 1 < rows || has_below) sv += fabsf(a - tile[i + W]);
    }
    acc_h += (double)sh;
    acc_v += (double)sv;
  }
  acc_h = warp_sum(acc_h);
  acc_v = warp_sum(acc_v);
  __shared__ double red[2][kTvThreads / 32];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { red[0][wid] = acc_h; red[1][wid] = acc_v; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, b = 0;
    for (int i = 0; i < kTvThreads / 32; ++i) { a += red[0][i]; b += red[1][i]; }
    atomicAdd(&sums[0], a);
    atomicAdd(&sums[1], b);
  }
}

__device__ __forceinline__ float sgnf(float v) { return (float)((v > 0.f) - (v < 0.f)); }

// dx_in (nullable): the gradient to accumulate onto, dx = dx_scale * dx_in + TV'; it may be dx itself (in place) and
// may have another element type than dx (a bf16 InfoNCE gradient under an fp32 x)
template <typename T, typename TI>
__global__ void __launch_bounds__(kTvThreads)
tv_bwd_kernel(const T* __restrict__ x, int64_t planes, int H, int W, int TH, const float* __restrict__ scale,
              T* dx, const TI* dx_in, const float* __restrict__ dx_scale) {
  extern __shared__ float tile[];  // [(TH+2)][W], row 0 = h0-1
  const int tiles_per_plane = (H + TH - 1) / TH;
  const int64_t n_tiles = planes * tiles_per_plane;
  const bool vec_ok = (W % 8 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  const float sh = scale[0], sv = scale[1];
  const float ds = (dx_scale != nullptr) ? dx_scale[0] : 1.f;
  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const int64_t pl = t / tiles_per_plane;
    const int h0 = (int)(t - pl * tiles_per_plane) * TH;
    const int rows = min(TH, H - h0);
    __syncthreads();
    tv_load_rows(x + pl * (int64_t)H * W, H, W, h0 - 1, rows + 2, tile, vec_ok);
    __syncthreads();
    T* out = dx + pl * (int64_t)H * W + (int64_t)h0 * W;
    const TI* in = dx_in ? dx_in + pl * (int64_t)H * W + (int64_t)h0 * W : nullptr;
    const float* ctr = tile + W;
    for (int i = threadIdx.x; i < rows * W; i += kTvThreads) {
      const int r = i / W, c = i - r * W;
      const int h = h0 + r;
      const float a = ctr[i];
      float g = 0.f;
      if (c + 1 < W) g += sh * sgnf(a - ctr[i + 1]);
      if (c >= 1) g -= sh * sgnf(ctr[i - 1] - a);
      if (h + 1 < H) g += sv * sgnf(a - ctr[i + W]);
      if (h >= 1) g -= sv * sgnf(ctr[i - W] - a);
      if (in) g += ds * ElemIO<TI>::ld(in + i);
      ElemIO<T>::st(out + i, g);
    }
  }
}


// ------------------------------------------------------------------------------------------------
// vectorised shared-memory tiled kernels (W % 8 == 0, 16-byte aligned base): the tile is filled with
// 16-byte cp.async copies in the tensor's own dtype; every thread then owns groups of 8 consecutive
// pixels of one row (one 16/32-byte shared load per row it touches).
// ------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void tv_fill_tile(const T* __restrict__ plane, int H, int W, int h_first, int n_rows, T* __restrict__ tile) {
  const int lo = h_first < 0 ? 0 : h_first;
  const int hi = (h_first + n_rows) > H ? H : (h_first + n_rows);
  if (hi > lo) {
    const char* src = reinterpret_cast<const char*>(plane + (int64_t)lo * W);
    char* dst = reinterpret_cast<char*>(tile + (int64_t)(lo - h_first) * W);
    const int bytes = (hi - lo) * W * (int)sizeof(T);
    for (int i = threadIdx.x * 16; i < bytes; i += kTvThreads * 16) {
      const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst + i);
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src + i) : "memory");
    }
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
}

__device__ __forceinline__ void lds8(const float* p, float (&v)[8]) {
  const float4 a = reinterpret_cast<const float4*>(p)[0], b = reinterpret_cast<const float4*>(p)[1];
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void lds8(const __nv_bfloat16* p, float (&v)[8]) {
  const uint4 r = *reinterpret_cast<const uint4*>(p);
  const uint32_t u[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) { v[2 * i] = __uint_as_float(u[i] << 16); v[2 * i + 1] = __uint_as_float(u[i] & 0xffff0000u); }
}
__device__ __forceinline__ float lds1(const float* p) { return *p; }
__device__ __forceinline__ float lds1(const __nv_bfloat16* p) { return __bfloat162float(*p); }

template <typename T>
__global__ void __launch_bounds__(kTvThreads)
tv_fwd_vec_kernel(const T* __restrict__ x, int64_t planes, int H, int W, int TH, double* __restrict__ sums) {
  extern __shared__ __align__(16) unsigned char tv_smem[];
  T* tile = reinterpret_cast<T*>(tv_smem);   // [(TH+1)][W]
  const int tiles_per_plane = (H + TH - 1) / TH;
  const int64_t n_tiles = planes * tiles_per_plane;
  const int gpr = W >> 3;   // groups of 8 pixels per row
  double acc_h = 0.0, acc_v = 0.0;
  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const int64_t pl = t / tiles_per_plane;
    const int h0 = (int)(t - pl * tiles_per_plane) * TH;
    const int rows = min(TH, H - h0);
    __syncthreads();
    tv_fill_tile(x + pl * (int64_t)H * W, H, W, h0, rows + 1, tile);
    __syncthreads();
    const bool has_below = (h0 + rows) < H;
    float sh = 0.f, sv = 0.f;
    for (int gi = threadIdx.x; gi < rows * gpr; gi += kTvThreads) {
      const int r = gi / gpr, c0 = (gi - r * gpr) << 3;
      const T* p = tile + r * W + c0;
      float v[8];
      lds8(p, v);
#pragma unroll
      for (int i = 0; i < 7; ++i) sh += fabsf(v[i] - v[i + 1]);
      if (c0 + 8 < W) sh += fabsf(v[7] - lds1(p + 8));
      if (r + 1 < rows || has_below) {
        float b[8];
        lds8(p + W, b);
#pragma unroll
        for (int i = 0; i < 8; ++i) sv += fabsf(v[i] - b[i]);
      }
    }
    acc_h += (double)sh;
    acc_v += (double)sv;
  }
  acc_h = warp_sum(acc_h);
  acc_v = warp_sum(acc_v);
  __shared__ double red[2][kTvThreads / 32];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { red[0][wid] = acc_h; red[1][wid] = acc_v; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, b = 0;
    for (int i = 0; i < kTvThreads / 32; ++i) { a += red[0][i]; b += red[1][i]; }
    atomicAdd(&sums[0], a);
    atomicAdd(&sums[1], b);
  }
}

template <typename T, typename TI>
__global__ void __launch_bounds__(kTvThreads)
tv_bwd_vec_kernel(const T* __restrict__ x, int64_t planes, int H, int W, int TH, const float* __restrict__ scale,
                  T* dx, const TI* dx_in, const float* __restrict__ dx_scale) {
  extern __shared__ __align__(16) unsigned char tv_smem[];
  T* tile = reinterpret_cast<T*>(tv_smem);   // [(TH+2)][W], row 0 = h0-1
  const int tiles_per_plane = (H + TH - 1) / TH;
  const int64_t n_tiles = planes * tiles_per_plane;
  const int gpr = W >> 3;
  const float sh = scale[0], sv = scale[1];
  const float ds = (dx_scale != nullptr) ? dx_scale[0] : 1.f;
  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const int64_t pl = t / tiles_per_plane;
    const int h0 = (int)(t - pl * tiles_per_plane) * TH;
    const int rows = min(TH, H - h0);
    __syncthreads();
    tv_fill_tile(x + pl * (int64_t)H * W, H, W, h0 - 1, rows + 2, tile);
    __syncthreads();
    T* out = dx + pl * (int64_t)H * W + (int64_t)h0 * W;
    const TI* in = dx_in ? dx_in + pl * (int64_t)H * W + (int64_t)h0 * W : nullptr;
    for (int gi = threadIdx.x; gi < rows * gpr; gi += kTvThreads) {
      const int r = gi / gpr, c0 = (gi - r * gpr) << 3;
      const int h = h0 + r;
      const T* p = tile + (r + 1) * W + c0;
      float v[8], g[8];
      lds8(p, v);
#pragma unroll
      for (int i = 0; i < 8; ++i) g[i] = 0.f;
#pragma unroll
      for (int i = 0; i < 7; ++i) {
        const float sg = sh * sgnf(v[i] - v[i + 1]);
        g[i] += sg;
        g[i + 1] -= sg;
      }
      if (c0 + 8 < W) g[7] += sh * sgnf(v[7] - lds1(p + 8));
      if (c0 > 0) g[0] -= sh * sgnf(lds1(p - 1) - v[0]);
      if (h + 1 < H) {
        float b[8];
        lds8(p + W, b);
#pragma unroll
        for (int i = 0; i < 8; ++i) g[i] += sv * sgnf(v[i] - b[i]);
      }
      if (h >= 1) {
        float a[8];
        lds8(p - W, a);
#pragma unroll
        for (int i = 0; i < 8; ++i) g[i] -= sv * sgnf(a[i] - v[i]);
      }
      T* o = out + r * W + c0;
      if (in) {
        float e[8];
        load8(in + r * W + c0, e);
#pragma unroll
        for (int i = 0; i < 8; ++i) g[i] = fmaf(ds, e[i], g[i]);
      }
      store8(o, g);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// bf16 inputs: packed bf16x2 arithmetic.  sign(a - b) of two bf16 values is formed from two packed compares
// (exact: no subtraction is rounded), the +-1 / 0 counts are exact in bf16, and only the final scale-and-add is
// rounded -- to the bf16 the gradient is stored in anyway.  ~10 instructions per element instead of ~30, which is
// what takes the bf16 kernels from instruction-bound to HBM-bound.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t bf2_sgn_diff(uint32_t a, uint32_t b) {     // sgn(a - b) per half, as bf16x2
  uint32_t g, l, d;
  asm("set.gt.bf16x2.bf16x2 %0, %1, %2;" : "=r"(g) : "r"(a), "r"(b));
  asm("set.lt.bf16x2.bf16x2 %0, %1, %2;" : "=r"(l) : "r"(a), "r"(b));
  asm("sub.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(g), "r"(l));
  return d;
}
__device__ __forceinline__ uint32_t bf2_sub(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("sub.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
__device__ __forceinline__ uint32_t bf2_mul_(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("mul.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
__device__ __forceinline__ uint32_t bf2_fma_(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("fma.rn.bf16x2 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
// (x1,x2),(x3,x4),... from pairs (x0,x1),(x2,x3),... and the pair to the right
__device__ __forceinline__ uint32_t bf2_shl1(uint32_t cur, uint32_t next) { return __byte_perm(cur, next, 0x5432); }

__global__ void __launch_bounds__(kTvThreads)
tv_bwd_bf16x2_kernel(const __nv_bfloat16* __restrict__ x, int64_t planes, int H, int W, int TH, const float* __restrict__ scale,
                     __nv_bfloat16* dx, const __nv_bfloat16* dx_in, const float* __restrict__ dx_scale) {
  extern __shared__ __align__(16) unsigned char tv_smem[];
  __nv_bfloat16* tile = reinterpret_cast<__nv_bfloat16*>(tv_smem);   // [(TH+2)][W], row 0 = h0-1
  const int tiles_per_plane = (H + TH - 1) / TH;
  const int64_t n_tiles = planes * tiles_per_plane;
  const int gpr = W >> 3;
  const uint32_t sh2 = pack_bf16x2(scale[0], scale[0]), sv2 = pack_bf16x2(scale[1], scale[1]);
  // the upstream scale of the accumulated gradient is applied as hi + lo bf16 parts (two fmas): 2^-17 relative
  const float ds = (dx_scale != nullptr) ? dx_scale[0] : 1.f;
  const float ds_hi = __bfloat162float(__float2bfloat16_rn(ds));
  const uint32_t dsh2 = pack_bf16x2(ds_hi, ds_hi), dsl2 = pack_bf16x2(ds - ds_hi, ds - ds_hi);
  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const int64_t pl = t / tiles_per_plane;
    const int h0 = (int)(t - pl * tiles_per_plane) * TH;
    const int rows = min(TH, H - h0);
    __syncthreads();
    tv_fill_tile(x + pl * (int64_t)H * W, H, W, h0 - 1, rows + 2, tile);
    __syncthreads();
    __nv_bfloat16* out = dx + pl * (int64_t)H * W + (int64_t)h0 * W;
    const __nv_bfloat16* in = dx_in ? dx_in + pl * (int64_t)H * W + (int64_t)h0 * W : nullptr;
    for (int gi = threadIdx.x; gi < rows * gpr; gi += kTvThreads) {
      const int r = gi / gpr, c0 = (gi - r * gpr) << 3;
      const int h = h0 + r;
      const __nv_bfloat16* p = tile + (r + 1) * W + c0;
      const uint4 cv = *reinterpret_cast<const uint4*>(p);
      const uint32_t c[4] = {cv.x, cv.y, cv.z, cv.w};
      // neighbours outside the plane are replaced by the pixel itself: sgn(0) = 0 drops the term
      const uint4 av = (h >= 1) ? *reinterpret_cast<const uint4*>(p - W) : cv;
      const uint4 bv = (h + 1 < H) ? *reinterpret_cast<const uint4*>(p + W) : cv;
      const uint32_t a[4] = {av.x, av.y, av.z, av.w}, b[4] = {bv.x, bv.y, bv.z, bv.w};
      const uint32_t left = (c0 > 0) ? (uint32_t)*reinterpret_cast<const unsigned short*>(p - 1) : (c[0] & 0xffffu);
      const uint32_t right = (c0 + 8 < W) ? (uint32_t)*reinterpret_cast<const unsigned short*>(p + 8) : (c[3] >> 16);
      uint32_t g[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint32_t xr = bf2_shl1(c[i], i < 3 ? c[i + 1] : right);                                 // right neighbours
        const uint32_t xl = (i > 0) ? __byte_perm(c[i - 1], c[i], 0x5432) : __byte_perm(left, c[0], 0x5410);   // left neighbours
        const uint32_t dh = bf2_sub(bf2_sgn_diff(c[i], xr), bf2_sgn_diff(xl, c[i]));
        const uint32_t dv = bf2_sub(bf2_sgn_diff(c[i], b[i]), bf2_sgn_diff(a[i], c[i]));
        g[i] = bf2_fma_(sv2, dv, bf2_mul_(sh2, dh));
      }
      uint4* o = reinterpret_cast<uint4*>(out + r * W + c0);
      if (in) {
        const uint4 ev = *reinterpret_cast<const uint4*>(in + r * W + c0);
        const uint32_t e[4] = {ev.x, ev.y, ev.z, ev.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) g[i] = bf2_fma_(dsl2, e[i], bf2_fma_(dsh2, e[i], g[i]));
      }
      *o = make_uint4(g[0], g[1], g[2], g[3]);
    }
  }
}

// (Measured, not adopted: |a - b| = max - min on packed words with the sums taken by `mma.sync.m16n8k16` against a
// constant +1/-1 B fragment -- 3 instead of ~10 instructions per element, results within 5e-8 of the oracle -- runs
// at 0.69 of HBM against 0.77: four legacy-path HMMAs per 256 elements per warp are more than the B200 sustains.)
// bf16 forward, column-strip walk: a thread owns one group of 8 pixels and walks down a strip of rows, so every
// row is unpacked once (the row below becomes the next centre) and there is no per-group index arithmetic --
// ~5 instructions per element instead of ~14 (the generic kernel above issues at 83 % of the scheduler peak).
__global__ void __launch_bounds__(kTvThreads)
tv_fwd_bf16_walk_kernel(const __nv_bfloat16* __restrict__ x, int64_t planes, int H, int W, int TH, double* __restrict__ sums) {
  extern __shared__ __align__(16) unsigned char tv_smem[];
  __nv_bfloat16* tile = reinterpret_cast<__nv_bfloat16*>(tv_smem);   // [(TH+1)][W]
  const int tiles_per_plane = (H + TH - 1) / TH;
  const int64_t n_tiles = planes * tiles_per_plane;
  const int gpr = W >> 3;                                  // groups of 8 pixels per row
  const int strips = max(1, kTvThreads / gpr);             // row strips per tile
  double acc_h = 0.0, acc_v = 0.0;
  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const int64_t pl = t / tiles_per_plane;
    const int h0 = (int)(t - pl * tiles_per_plane) * TH;
    const int rows = min(TH, H - h0);
    __syncthreads();
    tv_fill_tile(x + pl * (int64_t)H * W, H, W, h0, rows + 1, tile);
    __syncthreads();
    const bool has_below = (h0 + rows) < H;
    const int rps = (rows + strips - 1) / strips;          // rows per strip
    float sh[4] = {0.f, 0.f, 0.f, 0.f}, sv[4] = {0.f, 0.f, 0.f, 0.f};      // four independent accumulation chains each
    for (int task = threadIdx.x; task < gpr * strips; task += kTvThreads) {
      const int cg = task % gpr, strip = task / gpr;
      const int r0 = strip * rps, r1 = min(rows, r0 + rps);
      if (r0 >= r1) continue;
      const int c0 = cg << 3;
      const __nv_bfloat16* p = tile + r0 * W + c0;
      float v[8];
      lds8(p, v);
      for (int r = r0; r < r1; ++r, p += W) {
        const float right = (c0 + 8 < W) ? lds1(p + 8) : v[7];
#pragma unroll
        for (int i = 0; i < 7; ++i) sh[i & 3] += fabsf(v[i] - v[i + 1]);
        sh[3] += fabsf(v[7] - right);
        if (r + 1 < rows || has_below) {
          float b[8];
          lds8(p + W, b);
#pragma unroll
          for (int i = 0; i < 8; ++i) { sv[i & 3] += fabsf(v[i] - b[i]); v[i] = b[i]; }
        }
      }
    }
    acc_h += (double)((sh[0] + sh[1]) + (sh[2] + sh[3]));
    acc_v += (double)((sv[0] + sv[1]) + (sv[2] + sv[3]));
  }
  acc_h = warp_sum(acc_h);
  acc_v = warp_sum(acc_v);
  __shared__ double red[2][kTvThreads / 32];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { red[0][wid] = acc_h; red[1][wid] = acc_v; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, b = 0;
    for (int i = 0; i < kTvThreads / 32; ++i) { a += red[0][i]; b += red[1][i]; }
    atomicAdd(&sums[0], a);
    atomicAdd(&sums[1], b);
  }
}

// Rows too wide for a shared-memory tile (W > ~6000 f32 / ~12000 bf16 pixels): one thread per element, neighbours
// straight from global memory (L1 / L2 provide the reuse).  Same arithmetic and sign(0) = 0 as the tiled kernels.
template <typename T>
__global__ void __launch_bounds__(kTvThreads)
tv_fwd_direct_kernel(const T* __restrict__ x, int64_t planes, int H, int W, double* __restrict__ sums) {
  const int64_t n = planes * (int64_t)H * W;
  float sh = 0.f, sv = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % W);
    const int h = (int)((i / W) % H);
    const float a = ElemIO<T>::ld(x + i);
    if (c + 1 < W) sh += fabsf(a - ElemIO<T>::ld(x + i + 1));
    if (h + 1 < H) sv += fabsf(a - ElemIO<T>::ld(x + i + W));
  }
  double acc_h = warp_sum((double)sh), acc_v = warp_sum((double)sv);
  if ((threadIdx.x & 31) == 0) { atomicAdd(&sums[0], acc_h); atomicAdd(&sums[1], acc_v); }
}

template <typename T, typename TI>
__global__ void __launch_bounds__(kTvThreads)
tv_bwd_direct_kernel(const T* __restrict__ x, int64_t planes, int H, int W, const float* __restrict__ scale,
                     T* dx, const TI* dx_in, const float* __restrict__ dx_scale) {
  const int64_t n = planes * (int64_t)H * W;
  const float sh = scale[0], sv = scale[1];
  const float ds = (dx_scale != nullptr) ? dx_scale[0] : 1.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % W);
    const int h = (int)((i / W) % H);
    const float a = ElemIO<T>::ld(x + i);
    float g = 0.f;
    if (c + 1 < W) g += sh * sgnf(a - ElemIO<T>::ld(x + i + 1));
    if (c >= 1) g -= sh * sgnf(ElemIO<T>::ld(x + i - 1) - a);
    if (h + 1 < H) g += sv * sgnf(a - ElemIO<T>::ld(x + i + W));
    if (h >= 1) g -= sv * sgnf(ElemIO<T>::ld(x + i - W) - a);
    if (dx_in) g += ds * ElemIO<TI>::ld(dx_in + i);
    ElemIO<T>::st(dx + i, g);
  }
}

// Rows per tile.  The tile budget is in BYTES on the vector paths.  f32: 32-row tiles (33 KB, six resident blocks).  bf16
// is instruction-heavier per byte and does better with FEWER, LARGER tiles (each tile costs two block-wide barriers and
// a drained load pipeline): measured at 256 x 256 planes, forward 0.77 -> 0.87 of HBM with 128-row tiles (66 KB, opt-in
// shared memory, three resident blocks), backward 0.82 -> 0.85 and fused backward 0.85 -> 0.865 with 86-row tiles
// (48 KB); 64 KB+ tiles lose again on the backward.  Rows are balanced over the tiles of a plane (a plane is never
// split into two large tiles and a sliver).
static int tv_tile_rows(int H, int W, int halo, int elt_bytes, bool vec, bool fwd) {
  const bool big = vec && elt_bytes == 2;
  const int budget = (big && fwd) ? 66 * 1024 + 512 : kTvSmemFloats * 4;
  int r = (budget / elt_bytes) / W - halo;
  const int cap = big ? (fwd ? 128 : 94) : 32;
  if (r > cap) r = cap;
  if (r > H) r = H;
  if (r >= 1) {                        // balance: same number of tiles, equal heights
    const int n = (H + r - 1) / r;
    r = (H + n - 1) / n;
  }
  return r;
}
template <typename K>
static int tv_allow_smem(K kernel, size_t bytes, const char* what) {
  if (bytes <= 48 * 1024) return RC_OK;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) return fail(RC_ERR_CUDA, "%s: smem opt-in: %s", what, cudaGetErrorString(e));
  return RC_OK;
}

// ------------------------------------------------------------------------------------------------
// Smoothness backward from the difference signs the fused fp32 pre-pass kept (rc_infonce_prepass_tv: one word per 8-pixel
// group, pixel j at bits 4j .. 4j+3 = {sgn(x[h][w] - x[h][w+1]) + 1, sgn(x[h][w] - x[h+1][w]) + 1}, two bits each):
// dx = dx_scale * dx_in + sh * (c_h[w] - c_h[w-1]) + sv * (c_v[h] - c_v[h-1]) -- 0.5 bytes per element read instead of the
// fp32 x (the same arithmetic as tv_bwd_vec_kernel up to the order of the +-sh / +-sv additions).
// ------------------------------------------------------------------------------------------------
template <typename TI>
__global__ void __launch_bounds__(256)
tv_bwd_codes_kernel(const uint32_t* __restrict__ codes, int64_t planes, int H, int W, const float* __restrict__ scale,
                    float* __restrict__ dx, const TI* __restrict__ dx_in, const float* __restrict__ dx_scale) {
  const int gpr = W >> 3;
  const int64_t rows = planes * (int64_t)H;
  const float sh = scale[0], sv = scale[1];
  const float ds = (dx_scale != nullptr) ? dx_scale[0] : 1.f;
  constexpr uint32_t kLow2 = 0x33333333u, kNoDiff = 0x55555555u, kBias = 0x22222222u;
  // a warp per image row, lanes along its 8-pixel groups; the row's h is carried along the grid stride (a 64-bit
  // division per group made the first version of this kernel instruction bound)
  // (rows narrower than a warp: 32 / gpr rows per warp when that divides)
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  const int rpw = (gpr < 32 && 32 % gpr == 0) ? 32 / gpr : 1;
  const int lane_gi = rpw > 1 ? lane % gpr : lane, lane_row = rpw > 1 ? lane / gpr : 0;
  const int64_t row0 = ((int64_t)blockIdx.x * wpb + (threadIdx.x >> 5)) * rpw + lane_row, stride = (int64_t)gridDim.x * wpb * rpw;
  const int h_step = (int)(stride % H);
  int h = (int)(row0 % H);
  for (int64_t row = row0; row < rows; row += stride, h = (h + h_step >= H) ? h + h_step - H : h + h_step) {
    for (int gi = lane_gi; gi < gpr; gi += 32) {
      const int64_t g = row * gpr + gi;
      const uint32_t cw = __ldg(codes + g);
      const uint32_t lw = gi > 0 ? __ldg(codes + g - 1) : kNoDiff;          // no neighbour: code 1 = "no difference"
      const uint32_t aw = h > 0 ? __ldg(codes + g - gpr) : kNoDiff;
      float e[8], o[8];
      if (dx_in != nullptr) load8(dx_in + g * 8, e);
      // all eight pixels at once, one nibble each: (code - code of the previous pixel / the row above) + 2, in 0 .. 4
      const uint32_t hd = (cw & kLow2) + kBias - (((cw << 4) | ((lw >> 28) & 3u)) & kLow2);
      const uint32_t vd = ((cw >> 2) & kLow2) + kBias - ((aw >> 2) & kLow2);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float a = (float)((hd >> (4 * j)) & 15u) - 2.f;
        const float b = (float)((vd >> (4 * j)) & 15u) - 2.f;
        const float t = fmaf(sv, b, sh * a);
        o[j] = dx_in != nullptr ? fmaf(ds, e[j], t) : t;
      }
      store8(dx + g * 8, o);
    }
  }
}

}  // namespace rc

extern "C" int rc_tv_fwd(const void* x, rc_dtype x_dtype, int64_t planes, int H, int W, double* sums, void* stream) {
  RC_REQUIRE(x && sums, "rc_tv_fwd: null pointer");
  RC_REQUIRE(planes >= 0 && H >= 1 && W >= 1, "rc_tv_fwd: bad shape");
  if (planes == 0) return RC_OK;
  const bool vec = (W % 8 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  const int TH = rc::tv_tile_rows(H, W, 1, (vec && x_dtype != RC_F32) ? 2 : 4, vec, true);
  if (TH < 1) {          // wider than a shared-memory tile: element-wise kernel
    const int64_t n = planes * (int64_t)H * W;
    const int64_t nb = (n + rc::kTvThreads - 1) / rc::kTvThreads, capd = (int64_t)rc::num_sms() * 16;
    const int gridd = (int)(nb < capd ? nb : capd);
    if (x_dtype == RC_F32) rc::tv_fwd_direct_kernel<float><<<gridd, rc::kTvThreads, 0, (cudaStream_t)stream>>>((const float*)x, planes, H, W, sums);
    else rc::tv_fwd_direct_kernel<__nv_bfloat16><<<gridd, rc::kTvThreads, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x, planes, H, W, sums);
    return rc::check_launch("rc_tv_fwd(direct)");
  }
  const int64_t n_tiles = planes * ((H + TH - 1) / TH);
  const int64_t cap = (int64_t)rc::num_sms() * 8;
  const int grid = (int)(n_tiles < cap ? n_tiles : cap);
  const size_t smem = (size_t)(TH + 1) * W * sizeof(float);
  cudaStream_t s = (cudaStream_t)stream;
  if (vec) {
    const size_t vsmem = (size_t)(TH + 1) * W * (x_dtype == RC_F32 ? 4 : 2);
    int rcode = x_dtype == RC_F32 ? rc::tv_allow_smem(rc::tv_fwd_vec_kernel<float>, vsmem, "rc_tv_fwd") : rc::tv_allow_smem(rc::tv_fwd_bf16_walk_kernel, vsmem, "rc_tv_fwd");
    if (rcode) return rcode;
    if (x_dtype == RC_F32)
      rc::tv_fwd_vec_kernel<float><<<grid, rc::kTvThreads, vsmem, s>>>((const float*)x, planes, H, W, TH, sums);
    else
      rc::tv_fwd_bf16_walk_kernel<<<grid, rc::kTvThreads, vsmem, s>>>((const __nv_bfloat16*)x, planes, H, W, TH, sums);
  } else if (x_dtype == RC_F32)
    rc::tv_fwd_kernel<float><<<grid, rc::kTvThreads, smem, s>>>((const float*)x, planes, H, W, TH, sums);
  else
    rc::tv_fwd_kernel<__nv_bfloat16><<<grid, rc::kTvThreads, smem, s>>>((const __nv_bfloat16*)x, planes, H, W, TH, sums);
  return rc::check_launch("rc_tv_fwd");
}

// dx (x_dtype) = dx_scale * dx_in + scale_h d(sum_h)/dx + scale_v d(sum_v)/dx; dx_in nullable, any supported dtype pairing
static int tv_bwd_impl(const void* x, rc_dtype x_dtype, int64_t planes, int H, int W, const float* scale, void* dx,
                       const void* dx_in, rc_dtype in_dtype, const float* dx_scale, void* stream, const char* what) {
  using bf16 = __nv_bfloat16;
  RC_REQUIRE(x && dx && scale, "%s: null pointer", what);
  RC_REQUIRE(planes >= 0 && H >= 1 && W >= 1, "%s: bad shape", what);
  if (dx_in != nullptr && x_dtype == RC_BF16 && in_dtype != RC_BF16)
    return rc::fail(RC_ERR_UNSUPPORTED, "%s: an f32 dx_in needs an f32 x / dx", what);
  if (planes == 0) return RC_OK;
  const bool in_bf = dx_in != nullptr && in_dtype == RC_BF16;
  const bool vec = (W % 8 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) && ((reinterpret_cast<uintptr_t>(dx) & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(dx_in) & 15) == 0);
  const int TH = rc::tv_tile_rows(H, W, 2, (vec && x_dtype != RC_F32) ? 2 : 4, vec, false);
  cudaStream_t s = (cudaStream_t)stream;
  if (TH < 1) {          // wider than a shared-memory tile: element-wise kernel
    const int64_t n = planes * (int64_t)H * W;
    const int64_t nb = (n + rc::kTvThreads - 1) / rc::kTvThreads, capd = (int64_t)rc::num_sms() * 16;
    const int gridd = (int)(nb < capd ? nb : capd);
    if (x_dtype == RC_F32 && in_bf)
      rc::tv_bwd_direct_kernel<float, bf16><<<gridd, rc::kTvThreads, 0, s>>>((const float*)x, planes, H, W, scale, (float*)dx, (const bf16*)dx_in, dx_scale);
    else if (x_dtype == RC_F32)
      rc::tv_bwd_direct_kernel<float, float><<<gridd, rc::kTvThreads, 0, s>>>((const float*)x, planes, H, W, scale, (float*)dx, (const float*)dx_in, dx_scale);
    else
      rc::tv_bwd_direct_kernel<bf16, bf16><<<gridd, rc::kTvThreads, 0, s>>>((const bf16*)x, planes, H, W, scale, (bf16*)dx, (const bf16*)dx_in, dx_scale);
    return rc::check_launch(what);
  }
  const int64_t n_tiles = planes * ((H + TH - 1) / TH);
  const int64_t cap = (int64_t)rc::num_sms() * 8;
  const int grid = (int)(n_tiles < cap ? n_tiles : cap);
  const size_t smem = (size_t)(TH + 2) * W * sizeof(float);
  if (vec) {
    const size_t vsmem = (size_t)(TH + 2) * W * (x_dtype == RC_F32 ? 4 : 2);
    int rcode = x_dtype != RC_F32 ? rc::tv_allow_smem(rc::tv_bwd_bf16x2_kernel, vsmem, what)
                : in_bf        ? rc::tv_allow_smem(rc::tv_bwd_vec_kernel<float, bf16>, vsmem, what)
                               : rc::tv_allow_smem(rc::tv_bwd_vec_kernel<float, float>, vsmem, what);
    if (rcode) return rcode;
    if (x_dtype != RC_F32)
      rc::tv_bwd_bf16x2_kernel<<<grid, rc::kTvThreads, vsmem, s>>>((const bf16*)x, planes, H, W, TH, scale, (bf16*)dx, (const bf16*)dx_in, dx_scale);
    else if (in_bf)
      rc::tv_bwd_vec_kernel<float, bf16><<<grid, rc::kTvThreads, vsmem, s>>>((const float*)x, planes, H, W, TH, scale, (float*)dx, (const bf16*)dx_in, dx_scale);
    else
      rc::tv_bwd_vec_kernel<float, float><<<grid, rc::kTvThreads, vsmem, s>>>((const float*)x, planes, H, W, TH, scale, (float*)dx, (const float*)dx_in, dx_scale);
  } else if (x_dtype == RC_F32 && in_bf)
    rc::tv_bwd_kernel<float, bf16><<<grid, rc::kTvThreads, smem, s>>>((const float*)x, planes, H, W, TH, scale, (float*)dx, (const bf16*)dx_in, dx_scale);
  else if (x_dtype == RC_F32)
    rc::tv_bwd_kernel<float, float><<<grid, rc::kTvThreads, smem, s>>>((const float*)x, planes, H, W, TH, scale, (float*)dx, (const float*)dx_in, dx_scale);
  else
    rc::tv_bwd_kernel<bf16, bf16><<<grid, rc::kTvThreads, smem, s>>>((const bf16*)x, planes, H, W, TH, scale, (bf16*)dx, (const bf16*)dx_in, dx_scale);
  return rc::check_launch(what);
}

extern "C" int rc_tv_bwd(const void* x, rc_dtype x_dtype, int64_t planes, int H, int W, const float* scale,
                         void* dx, int accumulate, const float* dx_scale, void* stream) {
  return tv_bwd_impl(x, x_dtype, planes, H, W, scale, dx, accumulate ? dx : nullptr, x_dtype, dx_scale, stream, "rc_tv_bwd");
}

extern "C" int rc_tv_bwd_from(const void* x, rc_dtype x_dtype, int64_t planes, int H, int W, const float* scale,
                              const void* dx_in, rc_dtype dx_in_dtype, const float* dx_scale, void* dx_out, void* stream) {
  RC_REQUIRE(dx_in != nullptr, "rc_tv_bwd_from: null dx_in");
  return tv_bwd_impl(x, x_dtype, planes, H, W, scale, dx_out, dx_in, dx_in_dtype, dx_scale, stream, "rc_tv_bwd_from");
}

extern "C" int rc_tv_bwd_codes(const uint32_t* codes, int64_t planes, int H, int W, const float* scale, const void* dx_in,
                               rc_dtype dx_in_dtype, const float* dx_scale, float* dx_out, void* stream) {
  using bf16 = __nv_bfloat16;
  RC_REQUIRE(codes && scale && dx_out, "rc_tv_bwd_codes: null pointer");
  RC_REQUIRE(planes >= 0 && H >= 1 && W >= 1, "rc_tv_bwd_codes: bad shape");
  if (W % 8 != 0) return rc::fail(RC_ERR_UNSUPPORTED, "rc_tv_bwd_codes: W=%d must be a multiple of 8", W);
  RC_REQUIRE((reinterpret_cast<uintptr_t>(dx_out) & 15) == 0 && (reinterpret_cast<uintptr_t>(dx_in) & 15) == 0,
             "rc_tv_bwd_codes: dx_in / dx_out must be 16-byte aligned");
  if (planes == 0) return RC_OK;
  const int gpr = W / 8, rpw = (gpr < 32 && 32 % gpr == 0) ? 32 / gpr : 1;                   // a warp per row (or per 32 / gpr rows), 8 warps per block
  const int64_t nb = (planes * (int64_t)H + 8 * rpw - 1) / (8 * rpw), cap = (int64_t)rc::num_sms() * 16;
  const int grid = (int)(nb < cap ? nb : cap);
  cudaStream_t s = (cudaStream_t)stream;
  if (dx_in != nullptr && dx_in_dtype == RC_BF16)
    rc::tv_bwd_codes_kernel<bf16><<<grid, 256, 0, s>>>(codes, planes, H, W, scale, dx_out, (const bf16*)dx_in, dx_scale);
  else
    rc::tv_bwd_codes_kernel<float><<<grid, 256, 0, s>>>(codes, planes, H, W, scale, dx_out, (const float*)dx_in, dx_scale);
  return rc::check_launch("rc_tv_bwd_codes");
}
