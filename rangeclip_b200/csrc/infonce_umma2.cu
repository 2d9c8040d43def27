// K1/K2, CTA-pair version: the fused pixel-text InfoNCE forward + backward on
// `tcgen05.mma.cta_group::2`, software-pipelined across tiles.
//
// Two CTAs on neighbouring SMs form a cluster and work on two 128-pixel tiles at a time.  Every MMA
// spans both SMs (M = 256): each CTA stages only ITS half of the streamed operand and the tensor cores
// read the other half from the peer's shared memory, which halves the shared-memory fill traffic and
// the operand read traffic per SM:
//   S   = X^T T^T   M = 256 px (128 per CTA, A = own X tile, MN-major), N = Kp text rows, B split: Kp/2 rows per CTA
//   dX^T = T^T P^T   M = 256 channels (128 per CTA, A = own rows of T^T), N = 128 px (64 of each CTA's tile,
//                    B = own P rows), four [128 ch x 128 px] accumulators per tile pair per CTA
//
// Pipeline (per tile pair i; TMEM = S 256 columns + two 128-column dX accumulators, all 512 in use):
//   tensor pipe : S(0) | S(1) dX(0) | S(2) dX(1) | ...      S(i+1) is issued BEFORE dX(i)
//   softmax     : reads S(i) from TMEM while dX(i-1) runs, keeps P(i) = exp(z - m) as packed bf16 in
//                 REGISTERS, releases the S columns at once (so S(i+1) can start), and stores P(i) to the
//                 single shared-memory P buffer as soon as the dX(i-1) MMAs have finished reading P(i-1)
//   dX epilogue : own 128 channel rows x 64 contiguous pixels per accumulator: x is read straight from
//                 global memory (L2-resident: the S GEMM just streamed it) with 256-bit loads, prefetched one
//                 accumulator ahead; each warp stages its [32 d][32 px] dX box in shared memory and writes it
//                 with its own TMA store.
// Register budget by role (setmaxnreg; the sum over the five warpgroups must stay within the 5 x 96 the CTA is
// launched with): control warps 48, softmax warps 120, epilogue warps 96.
// Only the leader CTA (cluster rank 0) issues MMAs; completion is multicast to the mbarriers of both CTAs,
// consumer-release barriers live in the leader and receive remote arrivals from the peer.  The per-pixel
// row scales of a tile are exchanged through distributed shared memory (the dX epilogue of a CTA covers
// pixels of both tiles).
//
// This kernel runs forward-only launches, the dText path (it writes G for infonce_dt_umma.cu), rc_infonce_bf16_dyn and
// RC_INFONCE_SS_KERNEL; backward launches otherwise run the TS kernel (infonce_ts.cu), those of rc_infonce_bf16_dyn_kblock
// included.  The tiling, the operand
// producers, the relay and the softmax arithmetic are shared with it through infonce_pair.cuh, so that both give
// bit-identical dX and lse; this file holds the SS pipeline, the P store into shared memory (and the G store), the
// row-scale exchange between the CTAs and the dX epilogue.
#include "infonce_pair.cuh"

namespace rc {
using namespace umma;

namespace pair {
using namespace cta_pair;

constexpr int kThreads = 640;          // warps: 0 text TMA, 1 MMA (leader CTA only), 2 relay + TMEM alloc, 3 X TMA, 4-11 softmax, 12-19 dX epilogue
constexpr int kXStages = 4;            // X ring: own X chunks [64 d][128 px] (first touch: HBM latency; also read by the row norms)
constexpr int kTStages = 4;            // text ring: text half-chunks [Kp/2][64 d] for S, own T^T rows [128 d][64 k] for dX (L2 hits)
static_assert(kTStages >= 4, "a dX block keeps Kp/64 <= 4 slots of the text ring at once");
constexpr int kPBytes = 64 * 1024;
constexpr int kTmemCols = 512;
constexpr int kRegsCtl = 48, kRegsSoftmax = 120;     // epilogue warps keep the entry allocation (96); 48 + 2*120 + 2*96 = 5*96

struct __align__(8) Bars {
  uint64_t xf[kXStages];        // own X chunk has landed (CTA-local; relayed to the leader's xfull)
  uint64_t xfull[kXStages], xempty[kXStages];
  uint64_t tfull[kTStages], tempty[kTStages];
  uint64_t s_full[2], s_empty[2], p_full, p_empty;   // S: one TMEM buffer with a backward, two (columns 0 / 256) forward-only
  uint64_t acc_full[2], acc_empty[2];
  uint64_t sc_full[2];
  uint32_t tmem_base, pad;
};

constexpr int kOffT = kXStages * kStageBytes;
constexpr int kOffP = kOffT + kTStages * kStageBytes;
constexpr int kScaleBufs = 3;          // the softmax warps run up to two tiles ahead of the dX epilogue warps
constexpr int kOffScale = kOffP + kPBytes;                  // {rs, -cs} bf16x2 pairs: [kScaleBufs tiles][2 owner CTAs][64 px pairs] uint2
constexpr int kOffXch = kOffScale + 2 * kScaleBufs * 2 * 128 * 4;
constexpr int kOffStg = kOffXch + 2 * 4 * 2 * 128 * 4;      // exchange: [2 tile parities][max, sum, sez, sy][2 halves][128]
constexpr int kStgBytes = 32 * 32 * 2;                      // dX staging of one epilogue warp: [32 d][32 px] bf16, 64-byte swizzle
constexpr int kOffPart = kOffStg + 8 * kStgBytes;
constexpr int kOffBars = kOffPart + 8 * 128 * 4;            // row-norm partial sums of squares [8 softmax warps][128 px]
constexpr int kSmemBytes = kOffBars + (int)sizeof(Bars);
static_assert(kSmemBytes <= 232448, "shared-memory budget of one SM (227 KB)");

// bring-up ablation bits (Tiling::ablate): 1 no epilogue x loads, 2 no dX stores, 64 no row-norm reads, 128 no dX
// staging, 256 no text reloads
struct Params : Tiling {
  int store_g;              // 1: also write G = rs (P - sum onehot) (bf16 [B][HW][Kp]) for the dText GEMM
  int wide;                 // 1: rows of X / dX are 32-byte aligned (256-bit global accesses allowed)
  const __nv_bfloat16* x;
  // sync-free callers (device-side contrast-set builder, SURVEY 8f-2): the number of valid candidate rows and the log
  // temperature are read from device memory at kernel start (nullable: K / inv_tau above are used)
  const int32_t* k_dev;
  const float* log_tau_dev;
  int k0;                   // K-blocked launches with k_dev: first contrast row of this launch's block (block_rows)
};

// 16 pixels (32 bytes) of one channel row, straight from global memory.  `n8` = number of valid
// 8-pixel groups (0, 1 or 2); the 256-bit form needs 32-byte alignment (`wide`).
__device__ __forceinline__ void ldg_px16(const __nv_bfloat16* p, bool wide, int n8, uint32_t* r, uint64_t pol) {
  if (wide && n8 == 2 && pol != 0) {
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8], %9;"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "l"(p), "l"(pol));
  } else if (wide && n8 == 2) {
    asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "l"(p));
  } else {
#pragma unroll
    for (int g = 0; g < 2; ++g) {
      uint4 v = make_uint4(0, 0, 0, 0);
      if (g < n8) v = __ldg(reinterpret_cast<const uint4*>(p) + g);
      r[g * 4] = v.x; r[g * 4 + 1] = v.y; r[g * 4 + 2] = v.z; r[g * 4 + 3] = v.w;
    }
  }
}
// R = targets per embedding row (1, or 4 for the shared 2x2 form, see infonce_pair.cuh)
// kKB: K-blocked launches (Params::keep_w / lse_in); a template flag so that the headline instantiation carries none of it
template <bool kBwd, int R, bool kKB>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
infonce_umma_pair_kernel(const __grid_constant__ CUtensorMap map_x_s,   // X [B][D][HW], box (64 px, 64 d, 1)
                         const __grid_constant__ CUtensorMap map_t,     // T [Kp][D],    box (64 d, Kp/2 rows)
                         const __grid_constant__ CUtensorMap map_tt,    // T^T [D][Kp],  box (64 k, 128 d)
                         const __grid_constant__ CUtensorMap map_dx,    // dX [B][D][HW], box (32 px, 32 d, 1)
                         const __grid_constant__ CUtensorMap map_g,     // G [B][HW][Kp],  box (64 k, 128 px, 1) (dText only)
                         const Params prm) {
  extern __shared__ __align__(1024) uint8_t smem[];
  Bars* bars = reinterpret_cast<Bars*>(smem + kOffBars);
  uint32_t* sc_s = reinterpret_cast<uint32_t*>(smem + kOffScale);   // -cs as bf16x2 of a pixel PAIR: [kScaleBufs tiles][2 owner CTAs][64 pairs]
  const int lane = threadIdx.x & 31;
  const int warp = (int)(threadIdx.x >> 5);
  const uint32_t rank = cluster_ctarank();
  const bool leader_cta = rank == 0;
  constexpr bool kKbAll = kKB && R == 1;      // kb mode (rc_infonce_bf16_kblocks) exists for R = 1 only
  const int n_dchunks = prm.D / 64;      // 64-channel chunks of the S GEMM
  const int n_blk = prm.D / 256;         // 256-channel blocks of the dX GEMM
  const int n_kchunks = prm.Kp / 64;
  // MMA issue order per tile pair: the S GEMM of the next pair is split in two and wrapped around the dX blocks of
  // this pair, so that the dX epilogue drains accumulators while the tensor pipe works on S
  const int c_half = n_dchunks / 2;
  const int b_half = (n_blk + 1) / 2;
  const int n_clusters = gridDim.x / 2;
  const int cluster_id = blockIdx.x / 2;
  // an empty K block (rc_infonce_bf16_dyn_kblock): every CTA reads the same count, so the whole cluster leaves before any
  // barrier or tensor memory exists, and nothing is written
  if (kKB && prm.k_dev != nullptr && block_rows(prm.k_dev, prm.k0, prm.K) <= 0) return;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_x_s); tma_prefetch_desc(&map_t);
    if (kBwd) { tma_prefetch_desc(&map_tt); tma_prefetch_desc(&map_dx); }
    // X ring: xfull = the relays of both CTAs, xempty = MMA commit + the eight softmax warps (row norms);
    // text ring: tfull = the leader's expect_tx (bytes of both CTAs), tempty = MMA commit
    for (int i = 0; i < kXStages; ++i) { mbar_init(&bars->xf[i], 1); mbar_init(&bars->xfull[i], 2); mbar_init(&bars->xempty[i], 9); }
    for (int i = 0; i < kTStages; ++i) { mbar_init(&bars->tfull[i], 1); mbar_init(&bars->tempty[i], 1); }
    // consumer releases are ONE arrival per warp (after __syncwarp), not one per thread: an mbarrier arrive is a
    // shared-memory atomic, and 512 of them per hand-off (half of them remote) cost the leader's shared-memory pipe
    // more wavefronts than the P stores
    for (int i = 0; i < 2; ++i) { mbar_init(&bars->s_full[i], 1); mbar_init(&bars->s_empty[i], 16); }
    mbar_init(&bars->p_full, 16); mbar_init(&bars->p_empty, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&bars->acc_full[i], 1); mbar_init(&bars->acc_empty[i], 16); }
    mbar_init(&bars->sc_full[0], 5); mbar_init(&bars->sc_full[1], 5);   // 4 local writer warps + 1 expect_tx (peer: st.async)
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_2sm<kTmemCols>(&bars->tmem_base);
  if (kBwd) {
    for (int i = threadIdx.x; i < kPBytes / 16; i += kThreads) reinterpret_cast<uint4*>(smem + kOffP)[i] = make_uint4(0, 0, 0, 0);
    fence_proxy_async_smem();
  }
  tc_fence_before();
  cluster_sync();            // both CTAs' barriers are initialised before any remote arrive / 2-SM TMA credit
  tc_fence_after();
  const uint32_t tmem = bars->tmem_base;
#ifdef RC_TIMING
  long long wt[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) wt[i] = 0;
  const long long t_start = clock64();
#endif
  const uint32_t idesc_s = make_idesc_bf16(256, prm.Kp, /*A MN-major*/ 1, /*B K-major*/ 0);
  const uint32_t idesc_d = make_idesc_bf16(256, 128, 0, 0);

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsCtl));
    if (warp == 0 && lane == 0) {
      // =============================== TMA producer (both CTAs) ===============================
      // ring order == MMA issue order: S(first), then per tile pair [S(next)] [dX(this)]
      // text ring, in MMA issue order: S(first), then per tile pair
      //   [S(next) first half] [dX(this) first blocks] [S(next) second half] [dX(this) remaining blocks]
      uint32_t it = 0;
      auto koff_of = [&](int pj) -> int { return text_row0<kKbAll>(prm, pj); };
      auto load_s = [&](int c_begin, int c_end, int koff) {
        load_text_s<kTStages>(prm, &map_t, smem + kOffT, bars->tfull, bars->tempty, it, c_begin, c_end, koff, rank RC_WT);
      };
      auto load_dx = [&](int b_begin, int b_end, int koff) {
        for (int blk = b_begin; blk < b_end; ++blk)
          for (int kc = 0; kc < n_kchunks; ++kc, ++it) {   // own 128 rows of T^T for this 256-channel block, 64 k at a time
            const int st = it % kTStages;
            RC_WAIT(mbar_wait, &bars->tempty[st], ((it / kTStages) & 1) ^ 1, 2);
            if ((prm.ablate & 256) && it >= (uint32_t)kTStages) {
              if (leader_cta) mbar_arrive(&bars->tfull[st]);
              continue;
            }
            if (leader_cta) mbar_arrive_expect_tx(&bars->tfull[st], 2 * 16384);
            tma_load_2d_2sm(smem + kOffT + st * kStageBytes, &map_tt, &bars->tfull[st], koff + kc * 64, blk * 256 + (int)rank * 128);
          }
      };
      if (cluster_id < prm.n_pairs) load_s(0, n_dchunks, koff_of(cluster_id));
      for (int pj = cluster_id; pj < prm.n_pairs; pj += n_clusters) {
        const bool has_next = pj + n_clusters < prm.n_pairs;
        const int k_this = koff_of(pj), k_next = has_next ? koff_of(pj + n_clusters) : 0;
        if (has_next) load_s(0, c_half, k_next);
        if (kBwd) load_dx(0, b_half, k_this);
        if (has_next) load_s(c_half, n_dchunks, k_next);
        if (kBwd) load_dx(b_half, n_blk, k_this);
      }
    } else if (warp == 3 && lane == 0) {
      // =============================== X producer (both CTAs) ===============================
      // own X chunks of every tile, as far ahead as the X ring allows (the next tile's first chunks are in flight
      // while the dX GEMM of the previous pair runs)
      uint32_t xit = 0;
      for (int pj = cluster_id; pj < prm.n_pairs; pj += n_clusters)
        load_x_tile<kXStages, kKbAll, false>(prm, &map_x_s, smem, bars->xf, bars->xempty, xit, 2 * pj + (int)rank, n_dchunks, 0, 1 RC_WT);
    } else if (warp == 1 && leader_cta) {
      // =============================== MMA issuer (leader CTA) ================================
      // The whole warp runs the loop converged, so stage indices, addresses and descriptors live in uniform
      // registers; one elected lane issues the tcgen05 instructions.
      uint32_t it = 0, xit = 0, uc = 0;
      const uint32_t smem_base = smem_u32(smem);
      // descriptor templates: only the 14-bit start-address field changes (+ bytes/16 per step)
      const uint64_t dsc_x = desc_mnmajor_sw128(0, 8192);
      const uint64_t dsc_k = desc_kmajor_sw128(0);
      // S(n) goes to TMEM columns [0,256); forward-only launches alternate with [256,512) (no dX accumulators there),
      // so that the S GEMM of the next pair overlaps the softmax of this one
      auto issue_s = [&](uint32_t n, int c_begin, int c_end) {
        const uint32_t sidx = kBwd ? 0u : (n & 1u);
        const uint32_t s_tmem = tmem + sidx * 256;
        if (c_begin == 0) {
          RC_WAIT(mbar_wait, &bars->s_empty[sidx], (((kBwd ? n : (n >> 1)) & 1u) ^ 1u), 3);   // previous user has read it
          tc_fence_after();
        }
        for (int c = c_begin; c < c_end; ++c, ++it, ++xit) {
          const int sa = xit % kXStages, sb_ = it % kTStages;
          RC_WAIT(mbar_wait, &bars->xfull[sa], (xit / kXStages) & 1, 4);
          RC_WAIT(mbar_wait, &bars->tfull[sb_], (it / kTStages) & 1, 12);
          tc_fence_after();
          const uint64_t xa = dsc_x + ((smem_base + sa * kStageBytes) >> 4);
          const uint64_t tb = dsc_k + ((smem_base + kOffT + sb_ * kStageBytes) >> 4);
          if (elect_one()) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              mma_bf16_ss_2sm(s_tmem, xa + ((ks * 2048) >> 4), tb + ((ks * 32) >> 4), idesc_s, (c | ks) != 0);
            mma_commit_2sm(&bars->xempty[sa]);
            mma_commit_2sm(&bars->tempty[sb_]);
            if (c + 1 == n_dchunks) mma_commit_2sm(&bars->s_full[sidx]);
          }
          __syncwarp();
        }
      };
      const uint64_t pb = dsc_k + ((smem_base + kOffP) >> 4);
      uint32_t lt = 0;
      auto issue_dx = [&](int b_begin, int b_end) {
        for (int blk = b_begin; blk < b_end; ++blk) {
          for (int pxh = 0; pxh < 2; ++pxh, ++uc) {
            const int ab = uc & 1;
            RC_WAIT(mbar_wait, &bars->acc_empty[ab], ((uc >> 1) & 1) ^ 1, 6);
            tc_fence_after();
            if (blk < 2) RC_EV(lt, 3 + blk * 2 + pxh);     // dX unit issue starts (accumulator free; event ids 3-6)
            const uint32_t dcol = tmem + 256 + ab * 128;
            for (int kc = 0; kc < n_kchunks; ++kc) {
              const int st = (it + kc) % kTStages;
              if (pxh == 0) {          // the block's last text slot was requested only when the preceding S chunk retired:
                RC_WAIT(mbar_wait, &bars->tfull[st], ((it + kc) / kTStages) & 1, 7);     // wait per slot, not up front
                tc_fence_after();
              }
              const uint64_t sb = dsc_k + ((smem_base + kOffT + st * kStageBytes) >> 4);
              const uint64_t pk_ = pb + ((kc * 16384 + pxh * 8192) >> 4);
              if (elect_one()) {
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)     // A: own T^T rows [128 d][64 k]; B: own P rows [64 px][64 k]
                  mma_bf16_ss_2sm(dcol, sb + ((ks * 32) >> 4), pk_ + ((ks * 32) >> 4), idesc_d, (kc | ks) != 0);
                if (pxh == 1) mma_commit_2sm(&bars->tempty[st]);     // second (last) reader: the slot refills at once
              }
              __syncwarp();
            }
            if (elect_one()) mma_commit_2sm(&bars->acc_full[ab]);
            __syncwarp();
          }
          it += n_kchunks;
        }
      };
      if (cluster_id < prm.n_pairs) issue_s(0, 0, n_dchunks);
      for (int pj = cluster_id; pj < prm.n_pairs; pj += n_clusters, ++lt) {
        const bool has_next = pj + n_clusters < prm.n_pairs;
        if (has_next) {
          issue_s(lt + 1, 0, c_half);          // waits until the softmax warps have read the previous S out of these columns
          RC_EV(lt + 1, 0);        // S(lt+1) issue started
        }
        if (kBwd) {
          RC_WAIT(mbar_wait, &bars->p_full, lt & 1, 5);
          tc_fence_after();
          RC_EV(lt, 2);            // dX(lt) issue starts (P(lt) is in shared memory)
          issue_dx(0, b_half);
        }
        if (has_next) {
          issue_s(lt + 1, c_half, n_dchunks);
          RC_EV(lt + 1, 1);        // S(lt+1) issued
        }
        if (kBwd) {
          issue_dx(b_half, n_blk);
          if (elect_one()) mma_commit_2sm(&bars->p_empty);
          __syncwarp();
          RC_EV(lt, 7);            // dX(lt) issued
        }
      }
    }
    else if (warp == 2 && lane == 0) {
      // ========== relay (both CTAs): "own X chunk has landed" (CTA-local xf) -> the leader's full barrier ==========
      uint32_t xit = 0;
      for (int pj = cluster_id; pj < prm.n_pairs; pj += n_clusters)
        relay_x_tile<kXStages, true>(n_dchunks, bars->xf, bars->xfull, xit, leader_cta, 14 RC_WT);
    }
  } else if (warp < 12) {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegsSoftmax));
    // ======================= softmax / CE warps: own tile (two warps per TMEM lane quarter) =======================
    const int half = warp >= 8 ? 1 : 0;
    const int row = (warp & 3) * 32 + lane;                 // pixel of the own tile == TMEM lane
    const int Kh = prm.Kp >> 1;
    const int cb = half * Kh;
    const uint32_t trow0 = tmem + ((uint32_t)((warp & 3) * 32) << 16) + cb;
    uint8_t* prow = smem + kOffP + row * 128;
    const int sw = row & 7;
    float* xch_base = reinterpret_cast<float*>(smem + kOffXch);
    float loss_acc = 0.f, w_acc = 0.f, dlt_acc = 0.f;
    float gscale = 1.f, inv_wsum = 0.f;
    if (kBwd) grad_scales(prm, gscale, inv_wsum);
    float nx_ok, nx_w;         // pixel scalars of the next tile
    int nx_y;
    load_pixel_scalars<R>(prm, cluster_id < prm.n_pairs, 2 * cluster_id + (int)rank, row, nx_ok, nx_w, nx_y);
    // Row norms of the NEXT tile, computed by these warps while they would otherwise wait for its S GEMM
    float* part_s = reinterpret_cast<float*>(smem + kOffPart);
    int ng, nr;
    norm_coords(ng, nr);
    uint32_t nit = 0;
    float inv_n_next = 0.f;
    auto norm_next = [&]() {
      inv_n_next = norm_tile<kXStages>(smem, bars->xf, bars->xempty, nit, n_dchunks, part_s, warp, lane, row, ng, nr,
                                       (prm.ablate & 64) != 0, 15 RC_WT);
    };
    if (cluster_id < prm.n_pairs) norm_next();
    const float inv_tau = prm.log_tau_dev != nullptr ? expf(-__ldg(prm.log_tau_dev)) : prm.inv_tau;
    // rows past K_valid are zero pads; K-blocked launches with k_dev: the rows of their block (block_rows)
    const int K_valid = (kKB && prm.k_dev != nullptr) ? block_rows(prm.k_dev, prm.k0, prm.K)
                        : (prm.k_dev != nullptr ? max(1, min(__ldg(prm.k_dev), prm.K)) : prm.K);
    const bool use_bound = inv_tau * (2.02f * kLog2e) < 100.f;
    const float ml_bound = inv_tau * (1.01f * kLog2e);
    // peer copies of the row-scale arrays (same offsets in the other CTA's shared memory)
    const uint32_t sc_peer = map_to_cta(sc_s, rank ^ 1);
    const uint32_t sc_peer0 = map_to_cta(&bars->sc_full[0], rank ^ 1), sc_peer1 = map_to_cta(&bars->sc_full[1], rank ^ 1);
    uint32_t lt = 0;
    for (int pj = cluster_id; pj < prm.n_pairs; pj += n_clusters, ++lt) {
      const int tile = 2 * pj + (int)rank;
      const bool tile_ok = tile < prm.n_tiles;
      const int b = tile_ok ? div_tiles(prm, tile) : 0;
      const int px = tile_ok ? (tile - b * prm.tiles_per_img) * kTilePx + row : 0;
      const bool valid = tile_ok && px < prm.HW;
      // dText mode: the bulk store of the previous tile's G must have read the P buffer before anyone rewrites it
      // (every thread passes the named barrier below before its next P store)
      if (kBwd && prm.store_g && threadIdx.x == 128) tma_store_wait_read0();
      const int64_t m = (int64_t)b * prm.HW + px;
      // candidates in this tile's block (kb mode: the last block may be short; its zero pad rows are masked like any pad)
      const int Kt = (kKbAll && prm.kb > 0) ? min(256, prm.K - 256 * b) : K_valid;
      const float ok = nx_ok;
      const bool px_ok = ok != 0.f;
      const int yi = nx_y;
      const float wi = (R == 1 && (yi >= 0 || (kKB && prm.keep_w))) ? nx_w : 0.f;
      load_pixel_scalars<R>(prm, pj + n_clusters < prm.n_pairs, 2 * (pj + n_clusters) + (int)rank, row, nx_ok, nx_w, nx_y);
      float* xch = xch_base + (lt & 1) * (4 * 2 * 128);      // double-buffered: one named barrier per tile suffices
      const float inv_n = px_ok ? inv_n_next : 0.f;
      const float zs = inv_n * inv_tau;
      const float zl = zs * kLog2e;
      // forward-only: the tensor pipe runs one pair ahead (two S buffers), so the next tile's row norms are taken
      // first -- its X chunks are already streaming and their ring slots are refilled only after these reads
      if (!kBwd && pj + n_clusters < prm.n_pairs) norm_next();
      const uint32_t sidx = kBwd ? 0u : (lt & 1u);
      const uint32_t trow = trow0 + sidx * 256;
      RC_WAIT(mbar_wait, &bars->s_full[sidx], (kBwd ? lt : (lt >> 1)) & 1u, 8);
      tc_fence_after();
      if (warp == 4) RC_EV(lt, 10);    // S(lt) complete (seen by the softmax warps)
      RC_T0(tsm);
      const float ml = row_offset<kKB>(prm, valid, px, m, use_bound, ml_bound, trow, Kt, cb, Kh, xch, half, row, zl);
      // e = exp(z - m) for this half's columns; P stays in registers as packed bf16 until the P buffer is free
      uint32_t pk[64];
      float sy[R];
      float sum, sez;
      exp_pass<R>(trow, cb, Kh, Kt, yi, zl, ml, pk, sy, sum, sez);
      tc_fence_before();
      if (warp == 4) RC_EV(lt, 11);    // exp pass done
      if (warp == 11) RC_EV(lt, 15);   // exp pass done (last softmax warp)
      arrive_leader_warp(leader_cta, &bars->s_empty[sidx]);      // S columns are free: the tensor pipe may start the next S in them
      int yj[R];
      float wj[R];
      bool mine[R];
      float wtot, tz;
      gather_targets<R, kKB>(prm, yi, wi, ok, m, cb, Kh, sy, yj, wj, mine, wtot, tz);
      post_sums(xch, half, row, sum, sez, tz);
      named_bar_sync(2, 256);
      add_peer_sums(xch, half, row, sum, sez, tz);
      const float lse = row_lse<kKB>(prm, valid, ml, half, wtot, tz, zs, sum, loss_acc, w_acc);
      RC_TACC(1, tsm);
      if (!kBwd) {
        if (half == 0 && valid && prm.lse) prm.lse[m] = lse;
        continue;
      }
      {
        const float coefb = gscale * inv_wsum;      // formed per tile: kept live across the loop it costs time
        const float coef = coefb * wtot;
        const float inv_sum = 1.f / sum;
        const float rsv = p_scale(inv_n, inv_tau, coef, inv_sum);
        if (half == 0) {
          const float cj = proj_coef(coef, coefb, sez, tz, zs, inv_sum);
          const float csv = inv_n * inv_n * cj;
          // the dX epilogue works on packed bf16 pixel pairs: dx = acc + (-cs) * x
          const float cs_n = __shfl_down_sync(0xffffffffu, csv, 1);
          if ((lane & 1) == 0) {
            const uint32_t c2 = pack_bf16x2(-csv, -cs_n);
            const int idx = ((lt % kScaleBufs) * 2 + (int)rank) * 64 + (row >> 1);    // [tile buffer][owner = this CTA][pixel pair]
            sc_s[idx] = c2;
            st_async_remote_b32(sc_peer + idx * 4, c2, (lt & 1) ? sc_peer1 : sc_peer0);   // peer copy: 4 tx bytes on ITS barrier
          }
          dlt_acc -= cj;
          __syncwarp();
          if (lane == 0) mbar_arrive(&bars->sc_full[lt & 1]);                // own copy (one arrival per writer warp)
          if (row == 0) mbar_arrive_expect_tx(&bars->sc_full[lt & 1], 64 * 4);   // the peer's 64 st.async land here
        }
        // the dX MMAs of the previous pair have finished reading P: store this pair's P
        RC_WAIT(mbar_wait, &bars->p_empty, (lt & 1) ^ 1, 9);
        if (warp == 4) RC_EV(lt, 12);  // P buffer free
        RC_T0(tst);
        const uint32_t rs2 = pack_bf16x2(rsv, rsv);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (c * 32 < Kh) {
            const int k0 = cb + c * 32;
            uint8_t* sub = prow + (k0 >> 6) * 16384;
            const int cbase = (k0 & 32) >> 3;
#pragma unroll
            for (int g = 0; g < 4; ++g)
              *reinterpret_cast<uint4*>(sub + (((cbase + g) ^ sw) << 4)) =
                  make_uint4(bf2_mul(pk[c * 16 + g * 4], rs2), bf2_mul(pk[c * 16 + g * 4 + 1], rs2),
                             bf2_mul(pk[c * 16 + g * 4 + 2], rs2), bf2_mul(pk[c * 16 + g * 4 + 3], rs2));
          }
        }
        // the target entries of G, over the rounded P entries
#pragma unroll
        for (int j = 0; j < R; ++j) {
          if (mine[j]) {
            const float gv = target_g<R>(j, sy, yj, wj, wtot, sum, zl, ml, rsv);
            const int kk = yj[j] & 63;
            uint8_t* sub = prow + (yj[j] >> 6) * 16384;
            *reinterpret_cast<__nv_bfloat16*>(sub + (((kk >> 3) ^ sw) << 4) + (kk & 7) * 2) = __float2bfloat16_rn(gv);
          }
        }
        fence_proxy_async_smem();                 // P is read by the tensor cores (async proxy)
        arrive_leader_warp(leader_cta, &bars->p_full);
        if (warp == 4) RC_EV(lt, 13);  // P(lt) stored
        if (warp == 11) RC_EV(lt, 16); // P(lt) stored (last softmax warp)
        RC_TACC(2, tst);
        if (prm.store_g) {                        // dText: the finished G tile goes to global memory as it sits in smem
          named_bar_sync(6, 256);
          if (threadIdx.x == 128 && tile_ok) {
            const int gpx0 = px - row;
            for (int j = 0; j < n_kchunks; ++j) tma_store_3d(&map_g, smem + kOffP + j * 16384, j * 64, gpx0, b);
            tma_store_commit();
          }
        }
        if (half == 0 && valid && prm.lse && !(kKB && prm.lse_in != nullptr)) prm.lse[m] = lse;      // after the hand-off: nothing waits behind this store
        if (pj + n_clusters < prm.n_pairs) norm_next();
        if (warp == 4) RC_EV(lt, 14);  // row norms of the next tile done
      }
    }
    if (kBwd && prm.store_g && threadIdx.x == 128) tma_store_wait_all0();
    if (half == 0) add_sums<kBwd>(prm, lane, loss_acc, w_acc, dlt_acc);
  } else if (kBwd) {
    // ================ dX epilogue warps: own channel rows, 64 contiguous pixels per accumulator ================
    // Warps 12-15 (half 0) take accumulator columns [0,64) = pixels of CTA 0's tile, warps 16-19 (half 1) columns
    // [64,128) = pixels of CTA 1's tile; accumulator unit (blk, pxh) covers pixels [pxh*64, +64) of both tiles.
    const int half = warp >= 16 ? 1 : 0;
    const int row = (warp & 3) * 32 + lane;
    const uint32_t trow_acc = tmem + ((uint32_t)((warp & 3) * 32) << 16) + 256 + half * 64;
    const bool wide = prm.wide != 0;
    const int units_per_pair = n_blk * 2;
    // prefetch cursor: x of the NEXT 32-pixel chunk to be consumed from each of the two register buffers
    int f_pj = cluster_id, f_unit = 0;
    int64_t f_off = 0;        // element offset of (row, first pixel of the unit) in X
    int f_n8 = 0;             // valid 8-pixel groups in the 64-pixel span (0..8)
    int f_b = prm.B, f_px = 0, f_d = 0;   // TMA store coordinates of the unit (image index B = out of bounds: nothing is written)
    auto cursor_set = [&]() {
      f_n8 = 0; f_off = 0; f_b = prm.B; f_px = 0; f_d = 0;
      const int t = 2 * f_pj + half;
      if (f_pj < prm.n_pairs && t < prm.n_tiles) {
        const int b = div_tiles(prm, t);
        const int px0 = (t - b * prm.tiles_per_img) * kTilePx + (f_unit & 1) * 64;
        const int d = (f_unit >> 1) * 256 + (int)rank * 128 + row;
        f_b = b; f_px = px0; f_d = d - lane;
        f_off = ((int64_t)((kKbAll && prm.kb > 0) ? 0 : b) * prm.D + d) * prm.HW + px0;      // kb mode: X has one image
        const int64_t left = prm.HW - px0;
        f_n8 = left >= 64 ? 8 : (left > 0 ? (int)(left >> 3) : 0);
      }
    };
    auto cursor_next = [&]() {
      ++f_unit;
      if (f_unit >= units_per_pair) { f_unit = 0; f_pj += n_clusters; }
      cursor_set();
    };
    // Global accesses are made by lane PAIRS: lanes 2p, 2p+1 own channel rows 2p, 2p+1; access j of a 32-pixel chunk
    // touches row 2p+j, and lane b = lane & 1 moves the b-th 16-pixel (32-byte) piece -- so one warp instruction
    // covers 16 rows x 64 contiguous bytes instead of 32 rows x 32 bytes (half the L1 tag work).  A 2x2 exchange
    // inside the pair (pair_swap) turns "row 2p+j, piece b" into "own row, piece j" and back.
    const int lb = lane & 1;
    const uint64_t pol_x = l2_policy_evict_first();     // last use of these X lines in this kernel
    uint32_t xq[2][16];       // chunk c of the current unit; before pair_swap: [j][8] = (row 2p+j, piece b)
    auto pair_swap = [&](uint32_t* e) {
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const uint32_t send = lb ? e[r] : e[8 + r];
        const uint32_t recv = __shfl_xor_sync(0xffffffffu, send, 1);
        if (lb) e[r] = recv; else e[8 + r] = recv;
      }
    };
    auto fetch = [&](int c) {
      int n8 = min(2, max(0, f_n8 - (c * 2 + lb) * 2));      // valid 8-pixel groups of this lane's piece
      if (prm.ablate & 1) n8 = 0;
#pragma unroll
      for (int j = 0; j < 2; ++j)
        ldg_px16(prm.x + f_off + (int64_t)(j - lb) * prm.HW + c * 32 + lb * 16, wide, n8, &xq[c][j * 8], pol_x);
    };
    uint8_t* stg = smem + kOffStg + (warp - 12) * kStgBytes;
    const uint64_t pol_first = l2_policy_evict_first();  // dX is write-once: keep it from displacing X in L2
    cursor_set();
    fetch(0); fetch(1);
    uint32_t uc = 0, lt = 0;
    for (int pj = cluster_id; pj < prm.n_pairs; pj += n_clusters, ++lt) {
      RC_WAIT(mbar_wait, &bars->sc_full[lt & 1], (lt >> 1) & 1, 10);
      const uint32_t* sc = sc_s + (lt % kScaleBufs) * 128 + half * 64;
      for (int unit = 0; unit < units_per_pair; ++unit, ++uc) {
        const int ab = uc & 1;
        const int pxh = unit & 1;
        // where this unit's output goes (same cursor arithmetic as the prefetch, one unit behind)
        const int o_b = f_b, o_px = f_px, o_d = f_d;
        RC_WAIT(mbar_wait, &bars->acc_full[ab], (uc >> 1) & 1, 11);
        tc_fence_after();
        if (warp == 12) RC_EV(lt, 20 + unit * 2);      // accumulator of this unit complete
        RC_T0(tep);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          uint32_t acc[32];
          RC_T0(t3);
          tmem_ld_32x32(trow_acc + ab * 128 + c * 32, acc);
          tmem_ld_wait();
          RC_TACC(3, t3);
          RC_T0(t13);
          if (c == 1) { tc_fence_before(); arrive_leader_warp(leader_cta, &bars->acc_empty[ab]); }
          RC_TACC(13, t13);
          RC_T0(t4);
          pair_swap(&xq[c][0]);             // -> own row, pixels [c*32, +32) in order
          RC_TACC(4, t4);                   // first use of the prefetched x: exposed global-load latency shows here
          RC_T0(t7);
          const uint4* scp = reinterpret_cast<const uint4*>(sc + pxh * 32 + c * 16);    // -cs2 of 16 pixel pairs
          uint32_t o[16];
#pragma unroll
          for (int g = 0; g < 4; ++g) {       // four pixel pairs per step, packed bf16x2 arithmetic: dx = acc - cs x
            const uint4 sv = scp[g];
            const uint32_t cs4[4] = {sv.x, sv.y, sv.z, sv.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int i = 4 * g + j;
              const uint32_t a = pack_bf16x2(__uint_as_float(acc[2 * i]), __uint_as_float(acc[2 * i + 1]));
              o[i] = bf2_fma(cs4[j], xq[c][i], a);
            }
          }
          RC_TACC(7, t7);
          {
            // own row of the warp's [32 d][32 px] staging tile (64-byte swizzle), then one TMA store per warp
            RC_T0(t5);
            if (lane == 0) tma_store_wait_read0();           // the previous store has read the staging buffer
            __syncwarp();
            RC_TACC(5, t5);
            RC_T0(t8);
            uint8_t* srow = stg + lane * 64;
            const int sw64 = (lane >> 1) & 3;
#pragma unroll
            for (int g = 0; g < ((prm.ablate & 128) ? 0 : 4); ++g)
              *reinterpret_cast<uint4*>(srow + ((g ^ sw64) << 4)) = make_uint4(o[g * 4], o[g * 4 + 1], o[g * 4 + 2], o[g * 4 + 3]);
            RC_TACC(8, t8);
            RC_T0(t9);
            fence_proxy_async_smem();
            __syncwarp();
            RC_TACC(9, t9);
            RC_T0(t12);
            if (lane == 0 && !(prm.ablate & 2)) {
              if (kKB && prm.acc_dx) tma_reduce_add_3d(&map_dx, stg, o_px + c * 32, o_d, o_b);
              else tma_store_3d_hint(&map_dx, stg, o_px + c * 32, o_d, o_b, pol_first);
              tma_store_commit();
            }
            RC_TACC(12, t12);
          }
          // x of the NEXT unit's chunk c, into the registers this chunk has just released (both chunks of the next unit
          // are fetched relative to the advanced cursor)
          RC_T0(t6);
          if (c == 0) cursor_next();
          fetch(c);
          RC_TACC(6, t6);
        }
        RC_TACC(2, tep);
        if (warp == 12) RC_EV(lt, 21 + unit * 2);      // unit drained and stored
      }
    }
    if (lane == 0) tma_store_wait_all0();       // shared memory must stay valid until the last bulk store has read it
  }
#ifdef RC_TIMING
  if (prm.dbg != nullptr && blockIdx.x < 2 && lane == 0 && (warp == 0 || warp == 1 || warp == 4 || warp == 12)) {
    wt[0] = clock64() - t_start;
    const int role = warp == 0 ? 0 : (warp == 1 ? 1 : (warp == 4 ? 2 : 3));
#pragma unroll
    for (int i = 0; i < 16; ++i) prm.dbg[(blockIdx.x * 4 + role) * 16 + i] = wt[i];
  }
#endif
  tc_fence_before();
  cluster_sync();            // no CTA leaves while its peer may still touch its barriers / shared memory
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_2sm<kTmemCols>(tmem);
  }
}

}  // namespace pair

// D / 64 chunks of the S GEMM and D / 256 blocks of the dX GEMM (SS; TS: D / 64), whatever their number: the pipelines are
// tuned at D <= 512 and run unchanged at 768 and 1024 (CLIP ViT-L/14, ViT-H/14).  The X ring is shorter than a tile from
// D = 512 on, so the row norms and the S GEMM release its slots in turn (same chunk order, no other wait between them).
bool infonce_pair_supported(int D) { return D % 256 == 0 && D >= 256 && D <= 1024; }

// launch helper used by rc_infonce_bf16 (infonce.cu owns argument checking and the pre-pass)
int launch_infonce_pair(const InfoncePairArgs& a, cudaStream_t s) {
  using namespace pair;
  const bool bwd = a.dx != nullptr;
  CUtensorMap m_xs, m_t, m_tt, m_dx, m_g;
  int rcode;
  if ((rcode = make_operand_maps(a, 128, {"pair map_x_s", "pair map_t", "pair map_tt"}, &m_xs, &m_t, &m_tt))) return rcode;
  // dX [B][D][HW] (forward only: X again, unread)
  if ((rcode = make_xmap(&m_dx, bwd ? a.dx : a.xsrc, a, bwd || a.kb == 0 ? a.B : 1, 32, 32, "pair map_dx"))) return rcode;
  if (a.g_out != nullptr) {
    // G [B][HW][Kp] bf16: a tile is stored exactly as it sits in shared memory (four K-major 128B-swizzled sub-tiles)
    const int Kp = launch_kp(a);
    const uint64_t gdims[3] = {(uint64_t)Kp, (uint64_t)a.HW, (uint64_t)a.B};
    const uint64_t gstr[3] = {2, (uint64_t)Kp * 2, (uint64_t)a.HW * Kp * 2};
    const uint32_t gbox[3] = {64, 128, 1};
    if ((rcode = make_tmap_bf16(&m_g, a.g_out, 3, gdims, gstr, gbox, "pair map_g"))) return rcode;
  } else {
    m_g = m_dx;
  }
  Params prm;
  int grid = 0;
  if ((rcode = fill_tiling(prm, a, &grid))) return rcode;
  prm.store_g = a.g_out != nullptr;
  prm.wide = (a.HW % 16 == 0) && (reinterpret_cast<uintptr_t>(a.xsrc) % 32 == 0) && (reinterpret_cast<uintptr_t>(a.dx) % 32 == 0);
  prm.x = reinterpret_cast<const __nv_bfloat16*>(a.xsrc);
  prm.k_dev = a.k_dev; prm.log_tau_dev = a.log_tau_dev; prm.k0 = a.k0;
  auto launch = [&](auto kernel) -> int {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
    if (e != cudaSuccess) return fail(RC_ERR_CUDA, "rc_infonce_bf16(pair): smem opt-in: %s", cudaGetErrorString(e));
    kernel<<<grid, kThreads, kSmemBytes, s>>>(m_xs, m_t, m_tt, m_dx, m_g, prm);
    return check_launch("rc_infonce_bf16(pair)");
  };
  if (a.rep == 4) {
    if (launch_kblocked(a)) return bwd ? launch(infonce_umma_pair_kernel<true, 4, true>) : launch(infonce_umma_pair_kernel<false, 4, true>);
    return bwd ? launch(infonce_umma_pair_kernel<true, 4, false>) : launch(infonce_umma_pair_kernel<false, 4, false>);
  }
  if (launch_kblocked(a)) return bwd ? launch(infonce_umma_pair_kernel<true, 1, true>) : launch(infonce_umma_pair_kernel<false, 1, true>);
  return bwd ? launch(infonce_umma_pair_kernel<true, 1, false>) : launch(infonce_umma_pair_kernel<false, 1, false>);
}

}  // namespace rc
