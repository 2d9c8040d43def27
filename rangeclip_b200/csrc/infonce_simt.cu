// fp32 CUDA-core InfoNCE (forward + backward) and fp32 top-k logits: the full-precision path.
//
// Replaces model.py:272-291 (normalize, matmul, /tau, cross_entropy) and its autograd with one
// kernel that never materialises the [M, K] logits (parity gate: 1e-5 relative to the fp32
// reference).  The bf16 tensor-core kernels in infonce_umma.cu are the throughput path; this one
// also serves every shape they do not (K > 256, D % 64 != 0, tiny problems such as the area-image
// InfoNCE of model.py:304-321 with n <= batch size).
//
// Mapping: a block owns 32 consecutive pixel rows (lane = pixel, so global loads of the NCHW
// tensor are coalesced along HW); its 8 warps each own one eighth of the D channels in registers.
// Logits for 8 text rows at a time are reduced across the warps through shared memory.
// 512 < D <= 1024 (CLIP ViT-L/14, ViT-H/14): the wide form, 16 warps of 64 channels each, keeps the normalised pixel rows
// in shared memory instead ([D][32] fp32, lane = pixel: conflict-free) and only the dX accumulator in registers, so that
// 512 threads fit in 128 registers each.  Same arithmetic and accumulation order per warp slice.
#include "common.cuh"
#include <float.h>

namespace rc {

constexpr int kSimtThreads = 256;
constexpr int kSimtWarps = 8;
constexpr int kSimtKB = 8;   // text rows per exchange

template <int DPT>
struct SimtTile {
  float xh[DPT];     // normalised slice of this thread's pixel row
  float inv_norm;
  bool valid;        // pixel row exists
  int64_t off;       // element offset of x[b][slice_base][p]
};

template <int DPT>
__device__ __forceinline__ void simt_load_tile(SimtTile<DPT>& t, const float* __restrict__ x, int D, int64_t HW,
                                               int64_t ld_b, int64_t M, int64_t m, int slice, float (*red)[32]) {
  const int lane = threadIdx.x & 31;
  t.valid = m < M;
  const int64_t b = t.valid ? m / HW : 0;
  const int64_t p = t.valid ? m - b * HW : 0;
  t.off = b * ld_b + (int64_t)slice * DPT * HW + p;
  float ss = 0.f;
#pragma unroll
  for (int j = 0; j < DPT; ++j) {
    const int d = slice * DPT + j;
    const float v = (t.valid && d < D) ? __ldg(x + t.off + (int64_t)j * HW) : 0.f;
    t.xh[j] = v;
    ss = fmaf(v, v, ss);
  }
  red[slice][lane] = ss;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int s = 0; s < kSimtWarps; ++s) tot += red[s][lane];
  __syncthreads();
  const float nrm = fmaxf(sqrtf(tot), 1e-12f);   // F.normalize eps (model.py:273)
  t.inv_norm = 1.f / nrm;
#pragma unroll
  for (int j = 0; j < DPT; ++j) t.xh[j] = t.xh[j] / nrm;
}

// partial dots of this thread's slice against text rows k0..k0+7, exchanged through `part`
template <int DPT>
__device__ __forceinline__ void simt_logits(const SimtTile<DPT>& t, const float* __restrict__ text, int D, int K,
                                            int k0, int slice, float (*part)[kSimtKB][32], float scale,
                                            float (&z)[kSimtKB]) {
  const int lane = threadIdx.x & 31;
  float acc[kSimtKB];
#pragma unroll
  for (int kk = 0; kk < kSimtKB; ++kk) acc[kk] = 0.f;
  const int dbase = slice * DPT;
#pragma unroll
  for (int kk = 0; kk < kSimtKB; ++kk) {
    const int k = k0 + kk;
    if (k < K) {   // warp-uniform
      const float* row = text + (int64_t)k * D + dbase;
      if (dbase + DPT <= D) {
#pragma unroll
        for (int j = 0; j < DPT; j += 4) {
          const float4 tv = __ldg(reinterpret_cast<const float4*>(row + j));
          acc[kk] = fmaf(t.xh[j], tv.x, acc[kk]);
          acc[kk] = fmaf(t.xh[j + 1], tv.y, acc[kk]);
          acc[kk] = fmaf(t.xh[j + 2], tv.z, acc[kk]);
          acc[kk] = fmaf(t.xh[j + 3], tv.w, acc[kk]);
        }
      } else {
#pragma unroll
        for (int j = 0; j < DPT; ++j)
          if (dbase + j < D) acc[kk] = fmaf(t.xh[j], __ldg(row + j), acc[kk]);
      }
    }
  }
#pragma unroll
  for (int kk = 0; kk < kSimtKB; ++kk) part[slice][kk][lane] = acc[kk];
  __syncthreads();
#pragma unroll
  for (int kk = 0; kk < kSimtKB; ++kk) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kSimtWarps; ++w) s += part[w][kk][lane];
    z[kk] = s * scale;
  }
}

template <int DPT>
__global__ void __launch_bounds__(kSimtThreads, 1)
infonce_f32_kernel(const float* __restrict__ x, int B, int D, int64_t HW, int64_t ld_b,
                   const float* __restrict__ text, int K, const int32_t* __restrict__ y,
                   const float* __restrict__ w, float inv_tau, float* __restrict__ lse_out,
                   double* __restrict__ loss_sum, double* __restrict__ w_sum,
                   const double* __restrict__ w_sum_in, const float* __restrict__ grad_scale_p,
                   float* __restrict__ dx, float* __restrict__ dt, double* __restrict__ dlogtau) {
  __shared__ float red[kSimtWarps][32];
  __shared__ float part[2][kSimtWarps][kSimtKB][32];
  const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int64_t M = (int64_t)B * HW;
  const int64_t n_tiles = (M + 31) / 32;
  const bool need_bwd = (dx != nullptr) || (dt != nullptr) || (dlogtau != nullptr);
  double acc_loss = 0.0, acc_w = 0.0, acc_dlt = 0.0;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t m = tile * 32 + lane;
    SimtTile<DPT> t;
    simt_load_tile<DPT>(t, x, D, HW, ld_b, M, m, slice, red);
    const int yi = t.valid ? y[m] : -1;
    const float wi = (t.valid && yi >= 0) ? w[m] : 0.f;
    // ---- forward: online logsumexp over the K text rows
    float mx = -FLT_MAX, l = 0.f, zy = 0.f;
    int buf = 0;
    for (int k0 = 0; k0 < K; k0 += kSimtKB, buf ^= 1) {
      float z[kSimtKB];
      simt_logits<DPT>(t, text, D, K, k0, slice, part[buf], inv_tau, z);
      float bm = mx;
#pragma unroll
      for (int kk = 0; kk < kSimtKB; ++kk) if (k0 + kk < K) bm = fmaxf(bm, z[kk]);
      l *= expf(mx - bm);
#pragma unroll
      for (int kk = 0; kk < kSimtKB; ++kk)
        if (k0 + kk < K) {
          l += expf(z[kk] - bm);
          if (k0 + kk == yi) zy = z[kk];
        }
      mx = bm;
    }
    const float lse = mx + logf(l);
    if (slice == 0 && t.valid) {
      if (lse_out) lse_out[m] = lse;
      acc_loss += (double)(wi * (lse - zy));
      acc_w += (double)wi;
    }
    if (!need_bwd) continue;
    // ---- backward: recompute logits, dz = coef * (softmax - onehot)
    const double ws = w_sum_in[0];
    const float grad_scale = grad_scale_p ? grad_scale_p[0] : 1.f;
    const float coef = (ws > 0.0) ? grad_scale * wi / (float)ws : 0.f;
    float dxh[DPT];
#pragma unroll
    for (int j = 0; j < DPT; ++j) dxh[j] = 0.f;
    float c = 0.f;
    const int dbase = slice * DPT;
    __syncthreads();
    buf = 0;
    for (int k0 = 0; k0 < K; k0 += kSimtKB, buf ^= 1) {
      float z[kSimtKB];
      simt_logits<DPT>(t, text, D, K, k0, slice, part[buf], inv_tau, z);
#pragma unroll
      for (int kk = 0; kk < kSimtKB; ++kk) {
        const int k = k0 + kk;
        if (k < K) {
          const float pk = expf(z[kk] - lse);
          const float dz = coef * (pk - (k == yi ? 1.f : 0.f));
          c = fmaf(dz, z[kk], c);
          const float* row = text + (int64_t)k * D + dbase;
          if (dx != nullptr) {
#pragma unroll
            for (int j = 0; j < DPT; ++j)
              if (dbase + j < D) dxh[j] = fmaf(dz, __ldg(row + j), dxh[j]);
          }
          if (dt != nullptr) {
            const float dzs = dz * inv_tau;
#pragma unroll
            for (int j = 0; j < DPT; ++j) {
              const float s = warp_sum(dzs * t.xh[j]);
              if (lane == 0 && dbase + j < D && s != 0.f) atomicAdd(&dt[(int64_t)k * D + dbase + j], s);
            }
          }
        }
      }
    }
    if (dx != nullptr && t.valid) {
      // dx = (dxh/tau - xh * <xh, dxh/tau>) / |x|, with <xh, dxh/tau> = sum_k dz_k z_k = c  (Q2)
#pragma unroll
      for (int j = 0; j < DPT; ++j)
        if (dbase + j < D) dx[t.off + (int64_t)j * HW] = t.inv_norm * (inv_tau * dxh[j] - t.xh[j] * c);
    }
    if (slice == 0 && t.valid) acc_dlt -= (double)c;   // d z / d log(tau) = -z
  }
  if (slice == 0) {
    acc_loss = warp_sum(acc_loss);
    acc_w = warp_sum(acc_w);
    acc_dlt = warp_sum(acc_dlt);
    if (lane == 0) {
      if (loss_sum) atomicAdd(loss_sum, acc_loss);
      if (w_sum) atomicAdd(w_sum, acc_w);
      if (dlogtau && need_bwd) atomicAdd(dlogtau, acc_dlt);
    }
  }
}

// fp32 top-k over cosine logits (model.py:144,161-173); ties -> smaller reduced index (the index tie-break in the insertion
// keeps that order when a better value shifts the list down past equal entries).
template <int DPT>
__global__ void __launch_bounds__(kSimtThreads, 1)
eval_topk_f32_kernel(const float* __restrict__ x, int B, int D, int64_t HW, int64_t ld_b,
                     const float* __restrict__ text, int K, const int64_t* __restrict__ index_map, int k,
                     int64_t* __restrict__ out) {
  __shared__ float red[kSimtWarps][32];
  __shared__ float part[2][kSimtWarps][kSimtKB][32];
  const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int64_t M = (int64_t)B * HW;
  const int64_t n_tiles = (M + 31) / 32;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t m = tile * 32 + lane;
    SimtTile<DPT> t;
    simt_load_tile<DPT>(t, x, D, HW, ld_b, M, m, slice, red);
    float bv[8];
    int bi[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { bv[j] = -FLT_MAX; bi[j] = -1; }
    int buf = 0;
    for (int k0 = 0; k0 < K; k0 += kSimtKB, buf ^= 1) {
      float z[kSimtKB];
      simt_logits<DPT>(t, text, D, K, k0, slice, part[buf], 1.f, z);
#pragma unroll
      for (int kk = 0; kk < kSimtKB; ++kk) {
        if (k0 + kk < K) {
          float v = z[kk];
          int id = k0 + kk;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            // explicit index tie-break: a displaced entry moving down must pass equal values with larger indices
            if (j < k && (v > bv[j] || (v == bv[j] && (unsigned)id < (unsigned)bi[j]))) {
              const float tv = bv[j]; const int ti = bi[j];
              bv[j] = v; bi[j] = id; v = tv; id = ti;
            }
          }
        }
      }
    }
    if (slice == 0 && t.valid) {
      const int64_t b = m / HW, p = m - b * HW;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < k) out[(b * k + j) * HW + p] = bi[j] >= 0 ? index_map[bi[j]] : -1;
    }
  }
}

// ---- wide form: 512 < D <= 1024 --------------------------------------------------------------

constexpr int kWideWarps = 16;
constexpr int kWideThreads = kWideWarps * 32;
constexpr int kWideDPT = 64;                 // channels per warp slice
constexpr int kWideMaxD = kWideWarps * kWideDPT;
struct WideSmem {
  float xs[kWideMaxD][32];                   // normalised pixel rows of the tile: [channel][lane = pixel]
  float red[kWideWarps][32];
  float part[2][kWideWarps][kSimtKB][32];
};
constexpr int kWideSmemBytes = (int)sizeof(WideSmem);

// simt_load_tile with the slice in shared memory (each thread writes and reads only its own entries: no barrier between)
__device__ __forceinline__ void wide_load_tile(WideSmem& sm, const float* __restrict__ x, int D, int64_t HW, int64_t ld_b,
                                               int64_t M, int64_t m, int slice, float& inv_norm, bool& valid, int64_t& off) {
  const int lane = threadIdx.x & 31;
  valid = m < M;
  const int64_t b = valid ? m / HW : 0;
  const int64_t p = valid ? m - b * HW : 0;
  off = b * ld_b + (int64_t)slice * kWideDPT * HW + p;
  float ss = 0.f;
#pragma unroll 8
  for (int j = 0; j < kWideDPT; ++j) {
    const int d = slice * kWideDPT + j;
    const float v = (valid && d < D) ? __ldg(x + off + (int64_t)j * HW) : 0.f;
    sm.xs[slice * kWideDPT + j][lane] = v;
    ss = fmaf(v, v, ss);
  }
  sm.red[slice][lane] = ss;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int s = 0; s < kWideWarps; ++s) tot += sm.red[s][lane];
  __syncthreads();
  const float nrm = fmaxf(sqrtf(tot), 1e-12f);   // F.normalize eps (model.py:273)
  inv_norm = 1.f / nrm;
#pragma unroll 8
  for (int j = 0; j < kWideDPT; ++j) sm.xs[slice * kWideDPT + j][lane] = sm.xs[slice * kWideDPT + j][lane] / nrm;
}

// simt_logits with x̂ read from shared memory, in two steps: the slice partials into part[buf] (ends with a barrier), then
// the logit of row k0 + kk summed over the slices in warp order (wide_logit)
__device__ __forceinline__ void wide_partials(WideSmem& sm, const float* __restrict__ text, int D, int K, int k0, int slice,
                                              int buf) {
  const int lane = threadIdx.x & 31;
  float acc[kSimtKB];
#pragma unroll
  for (int kk = 0; kk < kSimtKB; ++kk) acc[kk] = 0.f;
  const int dbase = slice * kWideDPT;
  const float* xs = &sm.xs[dbase][lane];
  if (dbase + kWideDPT <= D) {
#pragma unroll 1
    for (int j = 0; j < kWideDPT; j += 4) {      // 8 text rows x 4 channels per step: 128 registers hold the dX slice too
      const float x0 = xs[j * 32], x1 = xs[(j + 1) * 32], x2 = xs[(j + 2) * 32], x3 = xs[(j + 3) * 32];
#pragma unroll
      for (int kk = 0; kk < kSimtKB; ++kk) {
        if (k0 + kk < K) {   // warp-uniform
          const float4 tv = __ldg(reinterpret_cast<const float4*>(text + (int64_t)(k0 + kk) * D + dbase + j));
          acc[kk] = fmaf(x0, tv.x, acc[kk]);
          acc[kk] = fmaf(x1, tv.y, acc[kk]);
          acc[kk] = fmaf(x2, tv.z, acc[kk]);
          acc[kk] = fmaf(x3, tv.w, acc[kk]);
        }
      }
    }
  } else if (dbase < D) {
#pragma unroll 1
    for (int j = 0; j < kWideDPT && dbase + j < D; ++j) {
      const float xv = xs[j * 32];
#pragma unroll
      for (int kk = 0; kk < kSimtKB; ++kk)
        if (k0 + kk < K) acc[kk] = fmaf(xv, __ldg(text + (int64_t)(k0 + kk) * D + dbase + j), acc[kk]);
    }
  }
#pragma unroll
  for (int kk = 0; kk < kSimtKB; ++kk) sm.part[buf][slice][kk][lane] = acc[kk];
  __syncthreads();
}
__device__ __forceinline__ float wide_logit(const WideSmem& sm, int buf, int kk, float scale) {
  const int lane = threadIdx.x & 31;
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < kWideWarps; ++w) s += sm.part[buf][w][kk][lane];
  return s * scale;
}
__device__ __forceinline__ void wide_logits(WideSmem& sm, const float* __restrict__ text, int D, int K, int k0, int slice,
                                            int buf, float scale, float (&z)[kSimtKB]) {
  wide_partials(sm, text, D, K, k0, slice, buf);
#pragma unroll
  for (int kk = 0; kk < kSimtKB; ++kk) z[kk] = wide_logit(sm, buf, kk, scale);
}

// infonce_f32_kernel at 512 < D <= 1024
__global__ void __launch_bounds__(kWideThreads, 1)
infonce_f32_wide_kernel(const float* __restrict__ x, int B, int D, int64_t HW, int64_t ld_b,
                        const float* __restrict__ text, int K, const int32_t* __restrict__ y,
                        const float* __restrict__ w, float inv_tau, float* __restrict__ lse_out,
                        double* __restrict__ loss_sum, double* __restrict__ w_sum,
                        const double* __restrict__ w_sum_in, const float* __restrict__ grad_scale_p,
                        float* __restrict__ dx, float* __restrict__ dt, double* __restrict__ dlogtau) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  WideSmem& sm = *reinterpret_cast<WideSmem*>(smem_raw);
  const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int64_t M = (int64_t)B * HW;
  const int64_t n_tiles = (M + 31) / 32;
  const bool need_bwd = (dx != nullptr) || (dt != nullptr) || (dlogtau != nullptr);
  double acc_loss = 0.0, acc_w = 0.0, acc_dlt = 0.0;
  const float* xs = &sm.xs[slice * kWideDPT][lane];
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t m = tile * 32 + lane;
    float inv_norm;
    bool valid;
    int64_t off;
    wide_load_tile(sm, x, D, HW, ld_b, M, m, slice, inv_norm, valid, off);
    const int yi = valid ? y[m] : -1;
    const float wi = (valid && yi >= 0) ? w[m] : 0.f;
    // ---- forward: online logsumexp over the K text rows
    float mx = -FLT_MAX, l = 0.f, zy = 0.f;
    int buf = 0;
    for (int k0 = 0; k0 < K; k0 += kSimtKB, buf ^= 1) {
      float z[kSimtKB];
      wide_logits(sm, text, D, K, k0, slice, buf, inv_tau, z);
      float bm = mx;
#pragma unroll
      for (int kk = 0; kk < kSimtKB; ++kk) if (k0 + kk < K) bm = fmaxf(bm, z[kk]);
      l *= expf(mx - bm);
#pragma unroll
      for (int kk = 0; kk < kSimtKB; ++kk)
        if (k0 + kk < K) {
          l += expf(z[kk] - bm);
          if (k0 + kk == yi) zy = z[kk];
        }
      mx = bm;
    }
    const float lse = mx + logf(l);
    if (slice == 0 && valid) {
      if (lse_out) lse_out[m] = lse;
      acc_loss += (double)(wi * (lse - zy));
      acc_w += (double)wi;
    }
    if (!need_bwd) { __syncthreads(); continue; }     // the next tile rewrites the rows and the exchange buffers
    // ---- backward: recompute logits, dz = coef * (softmax - onehot)
    const double ws = w_sum_in[0];
    const float grad_scale = grad_scale_p ? grad_scale_p[0] : 1.f;
    const float coef = (ws > 0.0) ? grad_scale * wi / (float)ws : 0.f;
    float dxh[kWideDPT];
#pragma unroll
    for (int j = 0; j < kWideDPT; ++j) dxh[j] = 0.f;
    float c = 0.f;
    const int dbase = slice * kWideDPT;
    __syncthreads();
    buf = 0;
    for (int k0 = 0; k0 < K; k0 += kSimtKB, buf ^= 1) {
      wide_partials(sm, text, D, K, k0, slice, buf);
#pragma unroll 1
      for (int kk = 0; kk < kSimtKB; ++kk) {
        const int k = k0 + kk;
        if (k < K) {
          const float zk = wide_logit(sm, buf, kk, inv_tau);
          const float pk = expf(zk - lse);
          const float dz = coef * (pk - (k == yi ? 1.f : 0.f));
          c = fmaf(dz, zk, c);
          const float* row = text + (int64_t)k * D + dbase;
          if (dx != nullptr) {
            if (dbase + kWideDPT <= D) {
#pragma unroll
              for (int j = 0; j < kWideDPT; j += 4) {
                const float4 tv = __ldg(reinterpret_cast<const float4*>(row + j));
                dxh[j] = fmaf(dz, tv.x, dxh[j]);
                dxh[j + 1] = fmaf(dz, tv.y, dxh[j + 1]);
                dxh[j + 2] = fmaf(dz, tv.z, dxh[j + 2]);
                dxh[j + 3] = fmaf(dz, tv.w, dxh[j + 3]);
              }
            } else {
#pragma unroll
              for (int j = 0; j < kWideDPT; ++j)
                if (dbase + j < D) dxh[j] = fmaf(dz, __ldg(row + j), dxh[j]);
            }
          }
          if (dt != nullptr) {
            const float dzs = dz * inv_tau;
#pragma unroll 4
            for (int j = 0; j < kWideDPT; ++j) {
              const float s = warp_sum(dzs * xs[j * 32]);
              if (lane == 0 && dbase + j < D && s != 0.f) atomicAdd(&dt[(int64_t)k * D + dbase + j], s);
            }
          }
        }
      }
    }
    if (dx != nullptr && valid) {
      // dx = (dxh/tau - xh * <xh, dxh/tau>) / |x|, with <xh, dxh/tau> = sum_k dz_k z_k = c  (Q2)
#pragma unroll
      for (int j = 0; j < kWideDPT; ++j)
        if (dbase + j < D) dx[off + (int64_t)j * HW] = inv_norm * (inv_tau * dxh[j] - xs[j * 32] * c);
    }
    if (slice == 0 && valid) acc_dlt -= (double)c;   // d z / d log(tau) = -z
    __syncthreads();
  }
  if (slice == 0) {
    acc_loss = warp_sum(acc_loss);
    acc_w = warp_sum(acc_w);
    acc_dlt = warp_sum(acc_dlt);
    if (lane == 0) {
      if (loss_sum) atomicAdd(loss_sum, acc_loss);
      if (w_sum) atomicAdd(w_sum, acc_w);
      if (dlogtau && need_bwd) atomicAdd(dlogtau, acc_dlt);
    }
  }
}

// eval_topk_f32_kernel at 512 < D <= 1024
__global__ void __launch_bounds__(kWideThreads, 1)
eval_topk_f32_wide_kernel(const float* __restrict__ x, int B, int D, int64_t HW, int64_t ld_b,
                          const float* __restrict__ text, int K, const int64_t* __restrict__ index_map, int k,
                          int64_t* __restrict__ out) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  WideSmem& sm = *reinterpret_cast<WideSmem*>(smem_raw);
  const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int64_t M = (int64_t)B * HW;
  const int64_t n_tiles = (M + 31) / 32;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t m = tile * 32 + lane;
    float inv_norm;
    bool valid;
    int64_t off;
    wide_load_tile(sm, x, D, HW, ld_b, M, m, slice, inv_norm, valid, off);
    float bv[8];
    int bi[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { bv[j] = -FLT_MAX; bi[j] = -1; }
    int buf = 0;
    for (int k0 = 0; k0 < K; k0 += kSimtKB, buf ^= 1) {
      float z[kSimtKB];
      wide_logits(sm, text, D, K, k0, slice, buf, 1.f, z);
#pragma unroll
      for (int kk = 0; kk < kSimtKB; ++kk) {
        if (k0 + kk < K) {
          float v = z[kk];
          int id = k0 + kk;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            // explicit index tie-break: a displaced entry moving down must pass equal values with larger indices
            if (j < k && (v > bv[j] || (v == bv[j] && (unsigned)id < (unsigned)bi[j]))) {
              const float tv = bv[j]; const int ti = bi[j];
              bv[j] = v; bi[j] = id; v = tv; id = ti;
            }
          }
        }
      }
    }
    if (slice == 0 && valid) {
      const int64_t b = m / HW, p = m - b * HW;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < k) out[(b * k + j) * HW + p] = bi[j] >= 0 ? index_map[bi[j]] : -1;
    }
    __syncthreads();                 // the next tile rewrites the rows
  }
}

// ---- small helpers ---------------------------------------------------------------------------

// one warp per text row: F.normalize (model.py:272 / :161), write f32 / bf16 / transposed bf16
__global__ void text_prepare_kernel(const float* __restrict__ text, int64_t ld_text, int64_t n_rows, const int64_t* __restrict__ idx,
                                    int K, int Kp, int D, float* __restrict__ t_f32, __nv_bfloat16* __restrict__ t_bf16,
                                    __nv_bfloat16* __restrict__ tt_bf16) {
  const int lane = threadIdx.x & 31;
  const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (k >= Kp) return;
  if (k >= K) {   // zero pad rows
    for (int d = lane; d < D; d += 32) {
      if (t_bf16) t_bf16[(int64_t)k * D + d] = __float2bfloat16_rn(0.f);
      if (tt_bf16) tt_bf16[(int64_t)d * Kp + k] = __float2bfloat16_rn(0.f);
    }
    return;
  }
  const int64_t src = idx ? idx[k] : (int64_t)k;
  if (src == -1) {   // pad entry of a device-built index list (rc_contrast_build): a zero row, like the rows past K
    for (int d = lane; d < D; d += 32) {
      if (t_f32) t_f32[(int64_t)k * D + d] = 0.f;
      if (t_bf16) t_bf16[(int64_t)k * D + d] = __float2bfloat16_rn(0.f);
      if (tt_bf16) tt_bf16[(int64_t)d * Kp + k] = __float2bfloat16_rn(0.f);
    }
    return;
  }
  if (src < 0 || src >= n_rows) {      // the reference raises an index error here (text[index_tensor]); a kernel cannot, and must not read out of bounds
    const float nan = __int_as_float(0x7fc00000);
    for (int d = lane; d < D; d += 32) {
      if (t_f32) t_f32[(int64_t)k * D + d] = nan;
      if (t_bf16) t_bf16[(int64_t)k * D + d] = __float2bfloat16_rn(nan);
      if (tt_bf16) tt_bf16[(int64_t)d * Kp + k] = __float2bfloat16_rn(nan);
    }
    return;
  }
  const float* row = text + src * ld_text;
  float ss = 0.f;
  for (int d = lane; d < D; d += 32) { const float v = row[d]; ss = fmaf(v, v, ss); }
  ss = warp_sum(ss);
  const float nrm = fmaxf(sqrtf(ss), 1e-12f);
  for (int d = lane; d < D; d += 32) {
    const float v = row[d] / nrm;
    if (t_f32) t_f32[(int64_t)k * D + d] = v;
    if (t_bf16) t_bf16[(int64_t)k * D + d] = __float2bfloat16_rn(v);
    if (tt_bf16) tt_bf16[(int64_t)d * Kp + k] = __float2bfloat16_rn(v);
  }
}

__global__ void weight_sum_kernel(const float* __restrict__ w, const int32_t* __restrict__ y, int64_t n,
                                  double* __restrict__ out) {
  double acc = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    if (y == nullptr || y[i] >= 0) acc += (double)w[i];
  acc = warp_sum(acc);
  __shared__ double red[8];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += red[i];
    if (s != 0.0) atomicAdd(out, s);
  }
}

// w starts as zeros; pass 1 counts multiplicities, pass 2 masks background and maps labels
__global__ void sample_count_kernel(const int64_t* __restrict__ rand_idx, int B, int64_t HW, int64_t n_samples,
                                    float* __restrict__ w) {
  const int64_t n = (int64_t)B * n_samples;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / n_samples;
    const int64_t p = rand_idx[i];
    if ((uint64_t)p < (uint64_t)HW) atomicAdd(&w[b * HW + p], 1.f);
  }
}
// counts[label] += 1 for every sampled pixel (label 0 and out-of-range labels included / skipped): the label histogram of
// model.py:222-226's gather, from which the set of sampled foreground labels follows without gathering or sorting them
__global__ void sample_label_count_kernel(const int64_t* __restrict__ seg, const int64_t* __restrict__ rand_idx, int B, int64_t HW,
                                          int64_t n_samples, int C, int32_t* __restrict__ counts) {
  extern __shared__ int32_t hist[];
  for (int i = threadIdx.x; i < C; i += blockDim.x) hist[i] = 0;
  __syncthreads();
  const int64_t n = (int64_t)B * n_samples;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / n_samples;
    const int64_t p = rand_idx ? rand_idx[i] : (i - b * n_samples);
    if ((uint64_t)p < (uint64_t)HW) {
      const int64_t lab = seg[b * HW + p];
      if ((uint64_t)lab < (uint64_t)C) atomicAdd(&hist[lab], 1);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += blockDim.x)
    if (hist[i] != 0) atomicAdd(&counts[i], hist[i]);
}
__global__ void sample_map_kernel(const int64_t* __restrict__ seg, int64_t n, const int32_t* __restrict__ map, int C,
                                  float* __restrict__ w, int32_t* __restrict__ y, int have_counts) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t lab = seg[i];
    int32_t yi = -1;
    if (lab > 0 && lab < C) yi = map[lab];          // model.py:226 drops label 0; :276-284 drops unmapped
    y[i] = yi;
    const float wi = have_counts ? w[i] : 1.f;
    w[i] = yi >= 0 ? wi : 0.f;
  }
}

// x *= s[0] in place, 16 bytes per thread per step; a scale of exactly one (W_text = 1, the reference default,
// model.py:337) leaves after reading the scalar, so the late upstream scaling of dX costs no pass over HBM
template <typename T>
__global__ void __launch_bounds__(256) scale_kernel(T* __restrict__ x, int64_t n, const float* __restrict__ s, int vec_ok) {
  const float f = s[0];
  if (f == 1.0f) return;
  constexpr int V = 16 / (int)sizeof(T);
  const int64_t nv = vec_ok ? n / V : 0;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = tid; i < nv; i += nt) {
    uint4 v = reinterpret_cast<uint4*>(x)[i];
    T* e = reinterpret_cast<T*>(&v);
#pragma unroll
    for (int j = 0; j < V; ++j) e[j] = static_cast<T>(static_cast<float>(e[j]) * f);     // registers: plain conversions
    reinterpret_cast<uint4*>(x)[i] = v;
  }
  for (int64_t i = nv * V + tid; i < n; i += nt) ElemIO<T>::st(x + i, ElemIO<T>::ld(x + i) * f);
}

// out = s[0] * x with a dtype conversion on the way (8 elements per thread per step): the late upstream scaling of a saved
// gradient into a FRESH buffer of the caller's dtype -- the saved tensor stays intact for a second backward
template <typename TI, typename TO>
__global__ void __launch_bounds__(256) scale_to_kernel(const TI* __restrict__ x, TO* __restrict__ out, int64_t n,
                                                        const float* __restrict__ s, int vec_ok) {
  const float f = s ? s[0] : 1.f;
  const int64_t nv = vec_ok ? n / 8 : 0;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = tid; i < nv; i += nt) {
    float v[8];
    load8(x + i * 8, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] *= f;
    store8(out + i * 8, v);
  }
  for (int64_t i = nv * 8 + tid; i < n; i += nt) ElemIO<TO>::st(out + i, ElemIO<TI>::ld(x + i) * f);
}

// grid: one block per SM, the wide form's shared memory opted in once per kernel
template <typename Kern>
static int wide_prepare(Kern kernel, const char* who) {
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kWideSmemBytes);
  if (e != cudaSuccess) return fail(RC_ERR_CUDA, "%s: smem opt-in: %s", who, cudaGetErrorString(e));
  return RC_OK;
}

template <template <int> class Launcher, typename... Args>
static int dispatch_dpt(int D, Args... args) {
  if (D <= 64) return Launcher<8>::run(args...);
  if (D <= 128) return Launcher<16>::run(args...);
  if (D <= 256) return Launcher<32>::run(args...);
  return Launcher<64>::run(args...);
}

template <int DPT> struct InfoNceLauncher {
  static int run(int grid, cudaStream_t s, const float* x, int B, int D, int64_t HW, int64_t ld_b, const float* t, int K,
                 const int32_t* y, const float* w, float inv_tau, float* lse, double* loss_sum, double* w_sum,
                 const double* w_sum_in, const float* grad_scale, float* dx, float* dt, double* dlogtau) {
    infonce_f32_kernel<DPT><<<grid, kSimtThreads, 0, s>>>(x, B, D, HW, ld_b, t, K, y, w, inv_tau, lse, loss_sum, w_sum,
                                                          w_sum_in, grad_scale, dx, dt, dlogtau);
    return 0;
  }
};
template <int DPT> struct TopkLauncher {
  static int run(int grid, cudaStream_t s, const float* x, int B, int D, int64_t HW, int64_t ld_b, const float* t, int K,
                 const int64_t* index_map, int k, int64_t* out) {
    eval_topk_f32_kernel<DPT><<<grid, kSimtThreads, 0, s>>>(x, B, D, HW, ld_b, t, K, index_map, k, out);
    return 0;
  }
};

}  // namespace rc

extern "C" int rc_infonce_f32(const float* x, int B, int D, int64_t HW, int64_t ld_b, const float* t, int K,
                              const int32_t* y, const float* w, float inv_tau, float* lse, double* loss_sum,
                              double* w_sum, const double* w_sum_in, const float* grad_scale, float* dx, float* dt,
                              double* dlogtau, void* stream) {
  RC_REQUIRE(x && t && y && w, "rc_infonce_f32: null pointer");
  RC_REQUIRE(B >= 0 && HW >= 0 && K >= 1, "rc_infonce_f32: bad shape");
  RC_REQUIRE(D >= 4 && D % 4 == 0, "rc_infonce_f32: D=%d must be a multiple of 4", D);
  if (D > rc::kWideMaxD) return rc::fail(RC_ERR_UNSUPPORTED, "rc_infonce_f32: D=%d is wider than %d", D, rc::kWideMaxD);
  RC_REQUIRE((reinterpret_cast<uintptr_t>(t) & 15) == 0, "rc_infonce_f32: text rows must be 16-byte aligned");
  if ((dx || dt || dlogtau) && !w_sum_in) return rc::fail(RC_ERR_INVALID, "rc_infonce_f32: gradients need w_sum_in");
  const int64_t M = (int64_t)B * HW;
  if (M == 0) return RC_OK;
  const int64_t tiles = (M + 31) / 32;
  const int64_t cap = (int64_t)rc::num_sms();
  const int grid = (int)(tiles < cap ? tiles : cap);
  if (D > 512) {
    int rcode = rc::wide_prepare(rc::infonce_f32_wide_kernel, "rc_infonce_f32");
    if (rcode) return rcode;
    rc::infonce_f32_wide_kernel<<<grid, rc::kWideThreads, rc::kWideSmemBytes, (cudaStream_t)stream>>>(
        x, B, D, HW, ld_b, t, K, y, w, inv_tau, lse, loss_sum, w_sum, w_sum_in, grad_scale, dx, dt, dlogtau);
    return rc::check_launch("rc_infonce_f32");
  }
  rc::dispatch_dpt<rc::InfoNceLauncher>(D, grid, (cudaStream_t)stream, x, B, D, HW, ld_b, t, K, y, w, inv_tau, lse,
                                        loss_sum, w_sum, w_sum_in, grad_scale, dx, dt, dlogtau);
  return rc::check_launch("rc_infonce_f32");
}

extern "C" int rc_eval_topk_f32(const float* x, int B, int D, int64_t HW, int64_t ld_b, const float* t, int K,
                                const int64_t* index_map, int k, int64_t* out, void* stream) {
  RC_REQUIRE(x && t && index_map && out, "rc_eval_topk_f32: null pointer");
  RC_REQUIRE(B >= 0 && HW >= 0 && K >= 1 && k >= 1 && k <= 8 && k <= K, "rc_eval_topk_f32: bad shape (k=%d K=%d)", k, K);
  RC_REQUIRE(D >= 4 && D % 4 == 0, "rc_eval_topk_f32: D=%d must be a multiple of 4", D);
  if (D > rc::kWideMaxD) return rc::fail(RC_ERR_UNSUPPORTED, "rc_eval_topk_f32: D=%d is wider than %d", D, rc::kWideMaxD);
  const int64_t M = (int64_t)B * HW;
  if (M == 0) return RC_OK;
  const int64_t tiles = (M + 31) / 32;
  const int64_t cap = (int64_t)rc::num_sms();
  const int grid = (int)(tiles < cap ? tiles : cap);
  if (D > 512) {
    int rcode = rc::wide_prepare(rc::eval_topk_f32_wide_kernel, "rc_eval_topk_f32");
    if (rcode) return rcode;
    rc::eval_topk_f32_wide_kernel<<<grid, rc::kWideThreads, rc::kWideSmemBytes, (cudaStream_t)stream>>>(
        x, B, D, HW, ld_b, t, K, index_map, k, out);
    return rc::check_launch("rc_eval_topk_f32");
  }
  rc::dispatch_dpt<rc::TopkLauncher>(D, grid, (cudaStream_t)stream, x, B, D, HW, ld_b, t, K, index_map, k, out);
  return rc::check_launch("rc_eval_topk_f32");
}

extern "C" int rc_text_prepare(const float* text, int64_t ld_text, int64_t n_rows, const int64_t* idx, int K, int D, float* t_f32,
                               void* t_bf16, void* tt_bf16, void* stream) {
  RC_REQUIRE(text && K >= 1 && D >= 1 && n_rows >= 1, "rc_text_prepare: bad argument");
  RC_REQUIRE(idx != nullptr || K <= n_rows, "rc_text_prepare: K=%d rows requested from a table of %lld", K, (long long)n_rows);
  const int Kp = (K + 63) / 64 * 64;
  const int rows = (t_bf16 || tt_bf16) ? Kp : K;
  rc::text_prepare_kernel<<<(rows + 3) / 4, 128, 0, (cudaStream_t)stream>>>(
      text, ld_text, n_rows, idx, K, rows, D, t_f32, (__nv_bfloat16*)t_bf16, (__nv_bfloat16*)tt_bf16);
  return rc::check_launch("rc_text_prepare");
}

extern "C" int rc_weight_sum(const float* w, const int32_t* y, int64_t n, double* w_sum, void* stream) {
  RC_REQUIRE(w && w_sum && n >= 0, "rc_weight_sum: bad argument");
  if (n == 0) return RC_OK;
  const int64_t blocks = (n + 255) / 256;
  const int grid = (int)(blocks < rc::num_sms() * 4 ? blocks : rc::num_sms() * 4);
  rc::weight_sum_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(w, y, n, w_sum);
  return rc::check_launch("rc_weight_sum");
}

extern "C" int rc_sample_weights(const int64_t* seg, const int64_t* rand_idx, int B, int64_t HW, int64_t n_samples,
                                 const int32_t* map, int C, float* w, int32_t* y, void* stream) {
  RC_REQUIRE(seg && map && w && y && B >= 0 && HW >= 0 && C >= 1, "rc_sample_weights: bad argument");
  const int64_t n = (int64_t)B * HW;
  if (n == 0) return RC_OK;
  cudaStream_t s = (cudaStream_t)stream;
  const int cap = rc::num_sms() * 8;
  if (rand_idx != nullptr) {
    cudaError_t e = cudaMemsetAsync(w, 0, (size_t)n * sizeof(float), s);
    if (e != cudaSuccess) return rc::fail(RC_ERR_CUDA, "rc_sample_weights: memset: %s", cudaGetErrorString(e));
    const int64_t ns = (int64_t)B * n_samples;
    if (ns > 0) {
      const int64_t blocks = (ns + 255) / 256;
      rc::sample_count_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, s>>>(rand_idx, B, HW, n_samples, w);
      int rcode = rc::check_launch("rc_sample_weights(count)");
      if (rcode) return rcode;
    }
  }
  const int64_t blocks = (n + 255) / 256;
  rc::sample_map_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, s>>>(seg, n, map, C, w, y, rand_idx != nullptr);
  return rc::check_launch("rc_sample_weights(map)");
}

extern "C" int rc_sample_label_counts(const int64_t* seg, const int64_t* rand_idx, int B, int64_t HW, int64_t n_samples, int C,
                                      int32_t* counts, void* stream) {
  RC_REQUIRE(seg && counts && B >= 0 && HW >= 0 && n_samples >= 0 && C >= 1, "rc_sample_label_counts: bad argument");
  if (C > 12000) return rc::fail(RC_ERR_UNSUPPORTED, "rc_sample_label_counts: C=%d labels exceed the shared-memory histogram", C);
  const int64_t ns = (int64_t)B * (rand_idx ? n_samples : HW);
  if (ns == 0) return RC_OK;
  const int64_t blocks = (ns + 1023) / 1024;
  const int cap = rc::num_sms() * 4;
  rc::sample_label_count_kernel<<<(int)(blocks < cap ? blocks : cap), 256, (size_t)C * 4, (cudaStream_t)stream>>>(
      seg, rand_idx, B, HW, rand_idx ? n_samples : HW, C, counts);
  return rc::check_launch("rc_sample_label_counts");
}

extern "C" int rc_scale(void* x, rc_dtype dtype, int64_t n, const float* sc, void* stream) {
  RC_REQUIRE(n >= 0, "rc_scale: bad argument");
  if (n == 0) return RC_OK;                       // an empty tensor has no storage to point at
  RC_REQUIRE(x && sc, "rc_scale: null pointer");
  const int64_t blocks = (n + 255) / 256;
  const int grid = (int)(blocks < rc::num_sms() * 8 ? blocks : rc::num_sms() * 8);
  const int vec_ok = (reinterpret_cast<uintptr_t>(x) & 15) == 0;
  if (dtype == RC_F32) rc::scale_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>((float*)x, n, sc, vec_ok);
  else rc::scale_kernel<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>((__nv_bfloat16*)x, n, sc, vec_ok);
  return rc::check_launch("rc_scale");
}

extern "C" int rc_scale_to(const void* x, rc_dtype x_dtype, void* out, rc_dtype out_dtype, int64_t n, const float* sc, void* stream) {
  using bf16 = __nv_bfloat16;
  RC_REQUIRE(n >= 0, "rc_scale_to: bad argument");
  if (n == 0) return RC_OK;
  RC_REQUIRE(x && out && x != out, "rc_scale_to: null pointer or in-place call (use rc_scale)");
  const int64_t blocks = (n / 8 + 255) / 256 + 1;
  const int grid = (int)(blocks < rc::num_sms() * 8 ? blocks : rc::num_sms() * 8);
  const int vec_ok = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out)) & 31) == 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (x_dtype == RC_BF16 && out_dtype == RC_BF16) rc::scale_to_kernel<bf16, bf16><<<grid, 256, 0, s>>>((const bf16*)x, (bf16*)out, n, sc, vec_ok);
  else if (x_dtype == RC_BF16) rc::scale_to_kernel<bf16, float><<<grid, 256, 0, s>>>((const bf16*)x, (float*)out, n, sc, vec_ok);
  else if (out_dtype == RC_BF16) rc::scale_to_kernel<float, bf16><<<grid, 256, 0, s>>>((const float*)x, (bf16*)out, n, sc, vec_ok);
  else rc::scale_to_kernel<float, float><<<grid, 256, 0, s>>>((const float*)x, (float*)out, n, sc, vec_ok);
  return rc::check_launch("rc_scale_to");
}
