// K1/K2, single-CTA version: the fused pixel-text InfoNCE forward + backward on the 5th-gen tensor cores (sm_100a).
// rc_infonce_bf16 runs it for D = 128 / 384 (the CTA-pair kernels in infonce_umma2.cu / infonce_ts.cu need D % 256 == 0).
//
// Replaces model.py:272-291 (normalize, [N,512]@[512,K], /tau, cross_entropy) and its autograd
// (CE backward, two matmuls, normalize backward, index_put/scatter_add).  Needs the pre-pass (rownorm_kernel,
// infonce.cu: 1/|x_p| and the bf16 copy of an fp32 X).  infonce_umma_kernel is persistent and warp-specialised; per
// 128-pixel tile
//   S  = X^T T^T           tcgen05.mma, A = X tile straight from NCHW (MN-major via TMA),
//                          B = text rows (K-major via TMA), fp32 accumulators in TMEM
//   softmax/CE epilogue    one thread per pixel reads its S row from TMEM: logsumexp, loss,
//                          dlogtau, and P = exp(z-m) - sum*onehot written as bf16 to smem
//   dX^T = T^T P^T         tcgen05.mma per 128-channel block, accumulators in TMEM
//   dX epilogue            row scale + normalize-backward projection, TMA store to NCHW
// The [B*HW, K] logits never leave the SM.
#include "common.cuh"
#include "umma.cuh"
#include "infonce_device.cuh"
#include <float.h>

namespace rc {

using namespace umma;

constexpr int kTilePx = 128;
constexpr int kThreads = 384;          // 12 warps: 0 TMA, 1 MMA, 2 TMEM alloc, 3 spare, 4-11 compute (softmax, then dX epilogue)
constexpr int kStages = 4;             // ring of 32 KB slots, each with its own full/empty barrier
constexpr int kStageBytes = 32 * 1024; // one slot = two X chunks (2 x 16 KB) | one text chunk (<= 32 KB) | T^T [128 d][<=128 k]
constexpr int kPBytes = 64 * 1024;     // P [128 px][<=256 k] bf16, four K-major 128B-swizzled sub-tiles
constexpr int kStgBufs = 3;             // dX staging buffers; X for the epilogue is prefetched kStgBufs-1 steps ahead
constexpr int kStgPx = 32;             // pixels per dX staging step
constexpr int kStgBytes = 128 * kStgPx * 2;   // [128 d][32 px] bf16 = 8 KB
constexpr int kTmemCols = 512;

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

// mbar_wait that also accumulates the cycles spent waiting (per role, reported for CTA 0)
#ifdef RC_TIMING
__device__ __forceinline__ void mbar_wait_t(uint64_t* bar, uint32_t parity, int tag, long long* acc) {
  const long long t0 = clock64();
  mbar_wait(bar, parity, tag);
  acc[tag] += clock64() - t0;
}
#else
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

// launch helper used by rc_infonce_bf16 (infonce.cu owns argument checking and the pre-pass)
int launch_infonce_1cta(const void* xsrc, void* dx, const void* t_bf16, const void* tt_bf16, int B, int D, int64_t HW, int K,
                        const float* inv_norm, const int32_t* y, const float* w, float inv_tau, const float* grad_scale,
                        const double* w_sum_in, float* lse, double* loss_sum, double* w_sum, double* dlogtau, cudaStream_t s) {
  const bool bwd = dx != nullptr;
  int rcode;
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
  prm.w_sum_in = w_sum_in; prm.lse = lse; prm.loss_sum = loss_sum; prm.w_sum = w_sum; prm.dlogtau = dlogtau; prm.dbg = debug_timing_buffer();
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

}  // namespace rc
