// K1/K2 with the softmax tile as a TENSOR-MEMORY operand (TS-mode tcgen05.mma) and TWO tile pairs in flight per CTA pair:
// the fused pixel-text InfoNCE forward + backward (model.py:272-291 and its autograd) for backward launches without dText.
// The tiling, the operand producers, the relay and the softmax arithmetic are shared with the SS kernel
// (infonce_umma2.cu) through infonce_pair.cuh, so that both give bit-identical dX and lse.  This file holds the TS
// pipeline (MMA issue order, tensor-memory slots), the P store into tensor memory and the dX epilogue.
//
// The SS kernel computes dX^T = T^T P^T with both operands in shared memory and keeps ONE S accumulator: the tensor
// pipe, the softmax warps and the dX epilogue wait for one another in a chain S(i) -> exp(i) -> P(i) -> dX(i), and the SS
// operand reads (96-128 B/clk) saturate the 128 B/clk shared-memory pipe.  Here
//   S  = X^T T^T    M = 256 px (128 per CTA; A = own X chunk [64 d][128 px], MN-major, shared memory), N = Kp,
//                   B = text rows split Kp/2 per CTA; fp32 accumulators in the 256 tensor-memory columns of a SLOT
//   P               the softmax threads overwrite the first 128 columns of the slot with the scaled softmax-minus-onehot
//                   tile as packed bf16 (tcgen05.st): P never touches shared memory
//   dX = P T        M = 256 px (the SAME TMEM lanes), A = P from tensor memory (TS mode), N = 64 channels per block,
//                   B = own 32 rows of T^T [D][Kp] (K-major, shared memory: 32 B/clk of operand reads); two 64-column fp32
//                   accumulators in the remaining 128 columns of the slot
// Tensor memory holds TWO slots (2 x 256 columns); tile pairs alternate between them.  MMA issue order
//   S(0) | dX(0)[0,2) S(1) dX(0)[2,n) | dX(1)[0,2) S(2) dX(1)[2,n) | ...      ([a,b): 64-channel blocks of dX)
// so the exp pass of pair j+1 runs while the tensor pipe works on dX(j) of the OTHER slot, and the dX epilogue drains the
// first two blocks of dX(j) while S(j+1) is computed: no role waits for a hand-off it has just produced.  Pixels stay on
// the TMEM lanes for both GEMMs, so a CTA's softmax and dX epilogue work on its own tile only (no row-scale exchange
// between the CTAs).  The dX epilogue thread owns a pixel: 32 channels per step come out of TMEM, the x values of the same
// [32 ch][32 px] box arrive by TMA in a small per-warp ring (the box doubles as the staging tile of the TMA store),
// dx = acc - cs x is formed in place and the box goes back with one TMA store.  The row norms 1/|x_p| are computed by the
// softmax warps from the X chunks in the operand ring.
#include "infonce_pair.cuh"

namespace rc {
using namespace umma;

namespace ts {
using namespace cta_pair;

constexpr int kThreads = 640;          // warps: 0 text TMA, 1 MMA (leader CTA), 2 relay + TMEM alloc, 3 X TMA, 4-11 softmax, 12-19 dX epilogue
constexpr int kXStages = 6;            // X ring: own X chunks [64 d][128 px]; deep, so that most of the next tile is resident early
constexpr int kTStages = 3;            // text ring: text half-chunks [Kp/2][64 d] for S, own T^T rows [32 ch][Kp] of a dX block
constexpr int kEpiBufs = 4;            // per epilogue warp: ring of [32 ch][32 px] bf16 boxes (x in, dX out)
constexpr int kEpiAhead = 2;           // x boxes requested this many steps ahead
constexpr int kEpiBufBytes = 2048;
constexpr int kTmemCols = 512;
constexpr int kSlotCols = 256;         // one slot: S [0,256) -> P [0,128) + two dX accumulators [128,192), [192,256)
constexpr int kColAcc = 128, kAccCols = 64;
constexpr int kDxLead = 2;             // dX blocks of pair l issued before S(l+1): one per accumulator of the slot
constexpr int kRegsCtl = 48, kRegsSoftmax = 120;     // epilogue warps keep the entry allocation (96); 48 + 2*120 + 2*96 = 5*96

struct __align__(8) Bars {
  uint64_t xf[kXStages];        // own X chunk has landed (CTA-local; relayed to the leader's xfull)
  uint64_t xfull[kXStages], xempty[kXStages];
  uint64_t tfull[kTStages], tempty[kTStages];
  uint64_t s_full[2], p_full[2];                  // per slot
  uint64_t acc_full[2][2], acc_empty[2][2];       // per slot, per accumulator
  uint64_t sc_full[4];                            // projection coefficients of a tile (by pair index & 3)
  uint64_t ebar[8][kEpiBufs];                     // x box of an epilogue warp has landed
  uint32_t tmem_base, pad;
};

constexpr int kScaleBufs = 4;          // the softmax warps run up to two tiles ahead of the dX epilogue warps
constexpr int kOffT = kXStages * kStageBytes;
constexpr int kOffEpi = kOffT + kTStages * kStageBytes;
constexpr int kOffScale = kOffEpi + 8 * kEpiBufs * kEpiBufBytes;      // -cs per pixel: [kScaleBufs][128] float
constexpr int kOffXch = kOffScale + kScaleBufs * 128 * 4;
constexpr int kOffPart = kOffXch + 2 * 4 * 2 * 128 * 4;               // exchange: [2 tile parities][max, sum, sez, sy][2 halves][128]
constexpr int kOffAcc = kOffPart + 8 * 128 * 4;                       // row-norm partial sums of squares [8 softmax warps][128 px]
constexpr int kOffBars = kOffAcc + 3 * 128 * 4;                       // per-pixel-row loss / weight / dlogtau sums [3][128]
constexpr int kSmemBytes = kOffBars + (int)sizeof(Bars);
static_assert(kSmemBytes <= 232448, "shared-memory budget of one SM (227 KB)");

// bring-up ablation bits (Tiling::ablate): 1 no epilogue x loads, 2 no dX stores, 256 no text reloads
// K-blocked launches of rc_infonce_bf16_dyn_kblock (read by the kKB instantiations only): the contrast set's valid rows and
// log(tau) in device memory (nullable: K and inv_tau are used), k0 = the first row of this launch's block (block_rows)
struct Params : Tiling {
  const int32_t* k_dev;
  const float* log_tau_dev;
  int k0;
};

// R = targets per embedding row (1, or 4 for the shared 2x2 form); kKB: K-blocked launches (keep_w / lse_in / kb)
template <int R, bool kKB>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
infonce_ts_kernel(const __grid_constant__ CUtensorMap map_x_s,   // X [B][D][HW], box (64 px, 64 d, 1), 128B swizzle
                  const __grid_constant__ CUtensorMap map_t,     // T [Kp][D],    box (64 d, Kp/2 rows)
                  const __grid_constant__ CUtensorMap map_tt,    // T^T [D][Kp],  box (64 k, 32 d)
                  const __grid_constant__ CUtensorMap map_xe,    // X [B][D][HW], box (32 px, 32 d, 1), 64B swizzle
                  const __grid_constant__ CUtensorMap map_dx,    // dX [B][D][HW], box (32 px, 32 d, 1), 64B swizzle
                  const Params prm) {
  extern __shared__ __align__(1024) uint8_t smem[];
  Bars* bars = reinterpret_cast<Bars*>(smem + kOffBars);
  float* sc_s = reinterpret_cast<float*>(smem + kOffScale);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader_cta = rank == 0;
  // kb mode (every candidate block in one launch, rc_infonce_bf16_kblocks) exists for R = 1 only; without this the
  // R = 4 K-blocked instantiation spills
  constexpr bool kKbAll = kKB && R == 1;
  const int n_dchunks = prm.D / 64;      // 64-channel chunks of the S GEMM
  const int n_blk = prm.D / 64;          // 64-channel blocks of the dX GEMM
  const int n_kchunks = prm.Kp / 64;
  const int n_clusters = gridDim.x / 2;
  const int cluster_id = blockIdx.x / 2;
  const int my_pairs = cluster_id < prm.n_pairs ? (prm.n_pairs - cluster_id + n_clusters - 1) / n_clusters : 0;
  // an empty K block: the whole cluster leaves before any barrier or tensor memory exists (infonce_umma2.cu); dX, lse and the
  // sums stay untouched, so an RC_INFONCE_ACCUMULATE_DX launch adds nothing
  if (kKB && prm.k_dev != nullptr && block_rows(prm.k_dev, prm.k0, prm.K) <= 0) return;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_x_s); tma_prefetch_desc(&map_t); tma_prefetch_desc(&map_tt);
    tma_prefetch_desc(&map_xe); tma_prefetch_desc(&map_dx);
    // X ring: xfull = the relays of both CTAs, xempty = MMA commit + the eight softmax warps (row norms)
    for (int i = 0; i < kXStages; ++i) { mbar_init(&bars->xf[i], 1); mbar_init(&bars->xfull[i], 2); mbar_init(&bars->xempty[i], 9); }
    for (int i = 0; i < kTStages; ++i) { mbar_init(&bars->tfull[i], 1); mbar_init(&bars->tempty[i], 1); }
    for (int sl = 0; sl < 2; ++sl) {
      mbar_init(&bars->s_full[sl], 1); mbar_init(&bars->p_full[sl], 16);     // consumer releases: one arrival per warp
      for (int ab = 0; ab < 2; ++ab) { mbar_init(&bars->acc_full[sl][ab], 1); mbar_init(&bars->acc_empty[sl][ab], 16); }
    }
    for (int i = 0; i < kScaleBufs; ++i) mbar_init(&bars->sc_full[i], 4);
    for (int i = 0; i < 8; ++i)
      for (int j = 0; j < kEpiBufs; ++j) mbar_init(&bars->ebar[i][j], 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_2sm<kTmemCols>(&bars->tmem_base);
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
  const uint32_t idesc_d = make_idesc_bf16(256, kAccCols, 0, 0);
  // l-th tile pair of this cluster
  auto pair_of = [&](int l) -> int { return cluster_id + l * n_clusters; };

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsCtl));
    if (warp == 0 && lane == 0) {
      // =============================== text producer (both CTAs) ===============================
      // ring order == MMA issue order: S(0) | dX(0)[0,2) S(1) dX(0)[2,n) | dX(1)[0,2) S(2) dX(1)[2,n) | ...
      uint32_t it = 0;
      auto load_s = [&](int l) {
        load_text_s<kTStages>(prm, &map_t, smem + kOffT, bars->tfull, bars->tempty, it, 0, n_dchunks,
                              text_row0<kKbAll>(prm, pair_of(l)), rank RC_WT);
      };
      auto load_dx = [&](int l, int b0, int b1) {     // per 64-channel block: own 32 rows of T^T, all Kp columns (4 KB per 64 k)
        const int koff = text_row0<kKbAll>(prm, pair_of(l));
        for (int blk = b0; blk < b1; ++blk, ++it) {
          const int st = it % kTStages;
          RC_WAIT(mbar_wait, &bars->tempty[st], ((it / kTStages) & 1) ^ 1, 2);
          if ((prm.ablate & 256) && it >= (uint32_t)kTStages) {
            if (leader_cta) mbar_arrive(&bars->tfull[st]);
            continue;
          }
          if (leader_cta) mbar_arrive_expect_tx(&bars->tfull[st], 2 * n_kchunks * 4096);
          for (int kc = 0; kc < n_kchunks; ++kc)
            tma_load_2d_2sm(smem + kOffT + st * kStageBytes + kc * 4096, &map_tt, &bars->tfull[st], koff + kc * 64,
                            blk * 64 + (int)rank * 32);
        }
      };
      if (my_pairs > 0) load_s(0);
      for (int l = 0; l < my_pairs; ++l) {
        load_dx(l, 0, kDxLead);
        if (l + 1 < my_pairs) load_s(l + 1);
        load_dx(l, kDxLead, n_blk);
      }
    } else if (warp == 3 && lane == 0) {
      // =============================== X producer (both CTAs) ===============================
      uint32_t xit = 0;
      // L2 policy of the two reads of a tile of X: the dX epilogue reads the tile again two pair iterations later, and in
      // between the L2 sees about 2 x 74 clusters x 256 KB of other X and as much dX written.  These loads mark the lines
      // evict_last and the epilogue's (last) load marks them evict_first, so that kept lines are released once consumed.
      const uint64_t pol_keep = l2_policy_evict_last();
      for (int l = 0; l < my_pairs; ++l)
        load_x_tile<kXStages, kKbAll, true>(prm, &map_x_s, smem, bars->xf, bars->xempty, xit, 2 * pair_of(l) + (int)rank, n_dchunks,
                                         pol_keep, 3 RC_WT);
    } else if (warp == 1 && leader_cta) {
      // =============================== MMA issuer (leader CTA) ================================
      // whole warp converged (addresses / descriptors in uniform registers), one elected lane issues
      uint32_t it = 0, xit = 0;
      uint32_t acc_par = 0;      // bit 2 * slot + accumulator: parity of that accumulator's launches so far (no local array)
      const uint32_t smem_base = smem_u32(smem);
      const uint64_t dsc_x = desc_mnmajor_sw128(0, 8192);
      const uint64_t dsc_k = desc_kmajor_sw128(0);
      // the slot's accumulators have been drained by the epilogue warps (all launches so far)
      auto wait_acc_free = [&](int sl, int ab, int tag) {
        RC_WAIT(mbar_wait, &bars->acc_empty[sl][ab], ((acc_par >> (2 * sl + ab)) & 1u) ^ 1u, tag);
      };
      auto issue_s = [&](int l) {
        const int sl = l & 1;
        const uint32_t s_tmem = tmem + sl * kSlotCols;
        // S overwrites the slot: its P has been consumed (the dX MMAs were issued before, the pipe runs in order) and
        // both dX accumulators must have been read out
        wait_acc_free(sl, 0, 7);
        wait_acc_free(sl, 1, 7);
        tc_fence_after();
        RC_EV(l, 0);               // S(l) issue starts (slot free)
        for (int c = 0; c < n_dchunks; ++c, ++it, ++xit) {
          const int sa = xit % kXStages, sb_ = it % kTStages;
          RC_WAIT(mbar_wait, &bars->xfull[sa], (xit / kXStages) & 1, 5);
          RC_WAIT(mbar_wait, &bars->tfull[sb_], (it / kTStages) & 1, 6);
          tc_fence_after();
          const uint64_t xa = dsc_x + ((smem_base + sa * kStageBytes) >> 4);
          const uint64_t tb = dsc_k + ((smem_base + kOffT + sb_ * kStageBytes) >> 4);
          if (elect_one()) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              mma_bf16_ss_2sm(s_tmem, xa + ((ks * 2048) >> 4), tb + ((ks * 32) >> 4), idesc_s, (c | ks) != 0);
            mma_commit_2sm(&bars->xempty[sa]);
            mma_commit_2sm(&bars->tempty[sb_]);
            if (c + 1 == n_dchunks) mma_commit_2sm(&bars->s_full[sl]);
          }
          __syncwarp();
        }
        RC_EV(l, 1);               // S(l) issued
      };
      auto issue_dx = [&](int l, int b0, int b1) {      // blocks [b0, b1) of dX(l)
        const int sl = l & 1;
        const uint32_t base = tmem + sl * kSlotCols;
        if (b0 == 0) {
          RC_WAIT(mbar_wait, &bars->p_full[sl], (l >> 1) & 1, 9);         // P(l) is in tensor memory
          tc_fence_after();
          RC_EV(l, 2);             // dX(l) issue starts (P(l) in tensor memory)
        }
        for (int blk = b0; blk < b1; ++blk, ++it) {
          const int ab = blk & 1;
          wait_acc_free(sl, ab, 4);
          if (blk < 8) RC_EV(l, 3 + blk);     // block's accumulator free
          const int st = it % kTStages;
          RC_WAIT(mbar_wait, &bars->tfull[st], (it / kTStages) & 1, 8);
          tc_fence_after();
          const uint64_t sb = dsc_k + ((smem_base + kOffT + st * kStageBytes) >> 4);
          const uint32_t dcol = base + kColAcc + ab * kAccCols;
          if (elect_one()) {
            for (int kc = 0; kc < n_kchunks; ++kc) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)     // A: P [256 px][16 k] in TMEM (8 columns); B: own T^T rows [32 ch][16 k]
                mma_bf16_ts_2sm(dcol, base + (kc * 4 + ks) * 8, sb + ((kc * 4096 + ks * 32) >> 4), idesc_d, (kc | ks) != 0);
            }
            mma_commit_2sm(&bars->tempty[st]);
            mma_commit_2sm(&bars->acc_full[sl][ab]);
          }
          __syncwarp();
          acc_par ^= 1u << (2 * sl + ab);
        }
        if (b1 == n_blk) RC_EV(l, 11);      // dX(l) issued
      };
      // S(l+1) goes between the first kDxLead blocks of dX(l) and the rest: the epilogue drains those blocks while the
      // tensor pipe computes S(l+1), instead of idling through every S GEMM
      if (my_pairs > 0) issue_s(0);
      for (int l = 0; l < my_pairs; ++l) {
        issue_dx(l, 0, kDxLead);
        if (l + 1 < my_pairs) issue_s(l + 1);
        issue_dx(l, kDxLead, n_blk);
      }
    } else if (warp == 2 && lane == 0) {
      // ========== relay (both CTAs): "own X chunk has landed" (CTA-local xf) -> the leader's full barrier ==========
      uint32_t xit = 0;
      for (int l = 0; l < my_pairs; ++l) relay_x_tile<kXStages, false>(n_dchunks, bars->xf, bars->xfull, xit, leader_cta, 10 RC_WT);
    }
  } else if (warp < 12) {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegsSoftmax));
    // ======================= softmax / CE warps: own tile (two warps per TMEM lane quarter) =======================
    const int half = warp >= 8 ? 1 : 0;
    const int row = (warp & 3) * 32 + lane;                 // pixel of the own tile == TMEM lane
    const int Kh = prm.Kp >> 1;
    const int cb = half * Kh;
    const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    float* xch_base = reinterpret_cast<float*>(smem + kOffXch);
    // the running loss / weight / dlogtau sums of a row live in shared memory: in registers they are spilled across the exp
    // pass (96 registers at compile time)
    float* acc_s = reinterpret_cast<float*>(smem + kOffAcc) + row;
    if (half == 0) acc_s[0] = acc_s[128] = acc_s[256] = 0.f;
    float gscale, inv_wsum;
    grad_scales(prm, gscale, inv_wsum);
    const float coefb = gscale * inv_wsum;
    float nx_ok, nx_w;         // pixel scalars of the next tile
    int nx_y;
    load_pixel_scalars<R>(prm, 0 < my_pairs, 2 * pair_of(0) + (int)rank, row, nx_ok, nx_w, nx_y);
    // Row norms: the X ring holds most of a tile, so its chunks are normally resident when they are taken, right before
    // the tile's exp pass.
    float* part_s = reinterpret_cast<float*>(smem + kOffPart);
    int ng, nr;
    norm_coords(ng, nr);
    uint32_t nit = 0;
    // log(tau) in device memory (kKB only): inv_tau formed as the SS kernel forms it, so that both stay bit-identical.  The
    // other instantiations read prm.inv_tau at every use, as they always have (a local copy changes their code).
    const float inv_tau_dev = (kKB && prm.log_tau_dev != nullptr) ? expf(-__ldg(prm.log_tau_dev)) : 0.f;
    auto inv_tau = [&]() { return (kKB && prm.log_tau_dev != nullptr) ? inv_tau_dev : prm.inv_tau; };
    const bool use_bound = inv_tau() * (2.02f * kLog2e) < 100.f;
    const float ml_bound = inv_tau() * (1.01f * kLog2e);
    for (int l = 0; l < my_pairs; ++l) {
      const int sl = l & 1;
      const int tile = 2 * pair_of(l) + (int)rank;
      const bool tile_ok = tile < prm.n_tiles;
      const int b = tile_ok ? div_tiles(prm, tile) : 0;
      const int px = tile_ok ? (tile - b * prm.tiles_per_img) * kTilePx + row : 0;
      const bool valid = tile_ok && px < prm.HW;
      const int64_t m = (int64_t)b * prm.HW + px;
      // valid candidate rows (rows past them are zero pads): kb mode's last block may be short; a block of
      // rc_infonce_bf16_dyn_kblock has block_rows of them
      const int Kt = (kKbAll && prm.kb > 0) ? min(256, prm.K - 256 * b)
                     : ((kKB && prm.k_dev != nullptr) ? block_rows(prm.k_dev, prm.k0, prm.K) : prm.K);
      const float ok = nx_ok;
      const bool px_ok = ok != 0.f;
      const int yi = nx_y;
      const float wi = (R == 1 && (yi >= 0 || (kKB && prm.keep_w))) ? nx_w : 0.f;
      load_pixel_scalars<R>(prm, l + 1 < my_pairs, 2 * pair_of(l + 1) + (int)rank, row, nx_ok, nx_w, nx_y);
      float* xch = xch_base + (l & 1) * (4 * 2 * 128);
      const uint32_t trow = lane_base + sl * kSlotCols + cb;
      RC_T0(tnorm);
      const float inv_n_tile = norm_tile<kXStages>(smem, bars->xf, bars->xempty, nit, n_dchunks, part_s, warp, lane, row, ng, nr, false,
                                                   11 RC_WT);
      RC_TACC(1, tnorm);
      if (warp == 4) RC_EV(l, 12);      // row norms of the tile done
      const float inv_n = px_ok ? inv_n_tile : 0.f;
      const float zs = inv_n * inv_tau();
      const float zl = zs * kLog2e;
      RC_WAIT(mbar_wait, &bars->s_full[sl], (l >> 1) & 1, 12);
      tc_fence_after();
      if (warp == 4) RC_EV(l, 13);      // S(l) complete (seen by the softmax warps)
      RC_T0(texp);
      const float ml = row_offset<kKB>(prm, valid, px, m, use_bound, ml_bound, trow, Kt, cb, Kh, xch, half, row, zl);
      uint32_t pk[64];
      float sy[R];
      float sum, sez;
      exp_pass<R>(trow, cb, Kh, Kt, yi, zl, ml, pk, sy, sum, sez);
      int yj[R];
      float wj[R];
      bool mine[R];
      float wtot, tz;
      gather_targets<R, kKB>(prm, yi, wi, ok, m, cb, Kh, sy, yj, wj, mine, wtot, tz);
      post_sums(xch, half, row, sum, sez, tz);
      // every softmax warp has read its S columns (tcgen05.wait::ld above): after this barrier the slot's columns may be
      // overwritten with P
      RC_TACC(2, texp);
      if (warp == 4) RC_EV(l, 14);      // exp pass done
      tc_fence_before();
      RC_T0(txch);
      named_bar_sync(2, 256);
      RC_TACC(13, txch);
      tc_fence_after();
      RC_T0(tpst);
      add_peer_sums(xch, half, row, sum, sez, tz);
      const float lse = row_lse<kKB>(prm, valid, ml, half, wtot, tz, zs, sum, acc_s[0], acc_s[128]);
      const float coef = coefb * wtot;
      const float inv_sum = 1.f / sum;
      const float rsv = p_scale(inv_n, inv_tau(), coef, inv_sum);
      if (half == 0) {
        const float cj = proj_coef(coef, coefb, sez, tz, zs, inv_sum);
        sc_s[(l & (kScaleBufs - 1)) * 128 + row] = -(inv_n * inv_n * cj);      // dx = acc + (-cs) x
        acc_s[256] -= cj;
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->sc_full[l & (kScaleBufs - 1)]);
      }
      {
        const uint32_t prow = lane_base + sl * kSlotCols + (cb >> 1);
        const uint32_t rs2 = pack_bf16x2(rsv, rsv);
        // the target entries of G, rounded to bf16, patched into the packed P words below
        uint32_t g16[R];
        int grel[R];
#pragma unroll
        for (int j = 0; j < R; ++j) {
          grel[j] = -1;
          g16[j] = 0;
          if (mine[j]) {
            const float gv = target_g<R>(j, sy, yj, wj, wtot, sum, zl, ml, rsv);
            grel[j] = yj[j] - cb;
            g16[j] = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(gv));
          }
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (c * 32 < Kh) {
            uint32_t v[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = bf2_mul(pk[c * 16 + i], rs2);
#pragma unroll
            for (int j = 0; j < R; ++j) {
              if (grel[j] >= 0 && (grel[j] >> 5) == c) {
                const int jj = (grel[j] >> 1) & 15;
                const bool hi = grel[j] & 1;
#pragma unroll
                for (int i = 0; i < 16; ++i)
                  if (i == jj) v[i] = hi ? ((v[i] & 0xffffu) | (g16[j] << 16)) : ((v[i] & 0xffff0000u) | g16[j]);
              }
            }
            tmem_st_32x16(prow + c * 16, v);
          }
        }
        tmem_st_wait();
        tc_fence_before();
        arrive_leader_warp(leader_cta, &bars->p_full[sl]);
      }
      RC_TACC(3, tpst);
      if (warp == 4) RC_EV(l, 15);      // P(l) stored
      if (half == 0 && valid && prm.lse && !(kKB && prm.lse_in != nullptr)) prm.lse[m] = lse;
    }
    if (half == 0) add_sums<true>(prm, lane, acc_s[0], acc_s[128], acc_s[256]);
  } else {
    // ================ dX epilogue warps: own tile, thread = pixel, one 64-channel block = one step of 32 channels ================
    // warp (q, h): TMEM lane quarter q = pixels [32 q, +32) of the tile, accumulator columns [32 h, +32) of every block
    const int ew = warp - 12;
    const int q = warp & 3, h = ew >> 2;
    uint8_t* ebuf = smem + kOffEpi + ew * (kEpiBufs * kEpiBufBytes);
    uint64_t* ebar = &bars->ebar[ew][0];
    const int total = my_pairs * n_blk;
    const uint64_t pol_first = l2_policy_evict_first();
    // cursor over (pair, block): coordinates of a step's box = (pixel, channel, image of x, image of dX)
    struct Cursor { int l, u, px, bo, bx; };
    auto cursor_pair = [&](Cursor& cu) {
      int b, px0;
      tile_coords(prm, 2 * pair_of(cu.l) + (int)rank, b, px0);
      cu.px = px0 + q * 32;
      cu.bo = b;
      cu.bx = (kKbAll && prm.kb > 0) ? (b < prm.B ? 0 : 1) : b;
    };
    auto cursor_next = [&](Cursor& cu) {
      if (++cu.u == n_blk) { cu.u = 0; ++cu.l; cursor_pair(cu); }
    };
    Cursor cs{0, 0, 0, 0, 0}, cr{0, 0, 0, 0, 0};      // step being stored / step being requested
    cursor_pair(cs);
    cursor_pair(cr);
    int s_req = 0;
    auto request_x = [&]() {                         // lane 0: the x box of step s_req
      const int bi = s_req % kEpiBufs;
      if (prm.ablate & 1) {           // bring-up: no x traffic (the box keeps stale data)
        mbar_arrive(&ebar[bi]);
        return;
      }
      mbar_arrive_expect_tx(&ebar[bi], kEpiBufBytes);
      // the tile's last read: release the lines the S GEMM's loads kept in the L2
      tma_load_3d_hint(ebuf + bi * kEpiBufBytes, &map_xe, &ebar[bi], cr.px, cr.u * 64 + h * 32, cr.bx, pol_first);
    };
    for (; s_req < kEpiAhead && s_req < total; ++s_req) {
      if (lane == 0) request_x();
      cursor_next(cr);
    }
    // The step works on 8x8 b16 matrices: tcgen05.ld.16x256b hands out the accumulators in the mma fragment layout (thread t:
    // pixel t/4 (+8), channel pair 2(t%4)), ldmatrix.trans reads x from the [32 ch][32 px] box (64-byte swizzle) in the SAME
    // layout and stmatrix.trans writes dX back over it -- ~40 instructions per thread and step instead of ~150 two-byte ones.
    // matrix (g, pb): channels [8g, +8) x pixels [8 pb, +8); one ldmatrix / stmatrix .x4 = the four pixel blocks of one g;
    // thread t addresses row (channel) 8g + (t & 7) of pixel block t >> 3
    const uint32_t moff = (uint32_t)((lane & 7) * 64 + ((((lane >> 3) ^ ((lane >> 1) & 3)) & 3) << 4));
    int s = 0;
    uint32_t acc_par = 0;      // bit 2 * slot + accumulator: parity of the completions seen so far
    for (int l = 0; l < my_pairs; ++l) {
      const int sl = l & 1;
      RC_WAIT(mbar_wait, &bars->sc_full[l & (kScaleBufs - 1)], (l >> 2) & 1, 14);
      uint32_t ncs2[4];                                // -cs of the thread's pixel in each of the four pixel blocks
#pragma unroll
      for (int pb = 0; pb < 4; ++pb) {
        const float v = sc_s[(l & (kScaleBufs - 1)) * 128 + q * 32 + pb * 8 + (lane >> 2)];
        ncs2[pb] = pack_bf16x2(v, v);
      }
      const uint32_t tacc = tmem + ((uint32_t)(q * 32) << 16) + sl * kSlotCols + kColAcc + h * 32;
      for (int blk = 0; blk < n_blk; ++blk, ++s) {
        const int ab = blk & 1;
        RC_WAIT(mbar_wait, &bars->acc_full[sl][ab], (acc_par >> (2 * sl + ab)) & 1u, 15);
        acc_par ^= 1u << (2 * sl + ab);
        tc_fence_after();
        if (warp == 12 && blk < 8) RC_EV(l, 20 + 2 * blk);      // block's accumulator complete
        RC_T0(tld);
        // accumulators of pixels [0,16) and [16,32) of the warp's lane quarter, 32 channel columns each, rounded to packed
        // bf16 channel pairs; the accumulator is handed back before any of it is processed
        uint32_t pa[4][4];                             // [g][pb]
        {
          uint32_t r[16];
          tmem_ld_16x256b_x4(tacc + ab * kAccCols, r);
          tmem_ld_wait();
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            pa[g][0] = pack_bf16x2(__uint_as_float(r[4 * g]), __uint_as_float(r[4 * g + 1]));
            pa[g][1] = pack_bf16x2(__uint_as_float(r[4 * g + 2]), __uint_as_float(r[4 * g + 3]));
          }
          tmem_ld_16x256b_x4(tacc + ab * kAccCols + (16u << 16), r);
          tmem_ld_wait();
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            pa[g][2] = pack_bf16x2(__uint_as_float(r[4 * g]), __uint_as_float(r[4 * g + 1]));
            pa[g][3] = pack_bf16x2(__uint_as_float(r[4 * g + 2]), __uint_as_float(r[4 * g + 3]));
          }
        }
        tc_fence_before();
        arrive_leader_warp(leader_cta, &bars->acc_empty[sl][ab]);
        RC_TACC(3, tld);
        const int bi = s % kEpiBufs;
        RC_WAIT(mbar_wait, &ebar[bi], (s / kEpiBufs) & 1, 4);
        RC_T0(tmath);
        // dx = acc - cs x in place on the box (same rounding as infonce_umma2.cu: the accumulator is rounded to bf16, then
        // one fused multiply-add on packed pairs)
        const uint32_t bx0 = smem_u32(ebuf + bi * kEpiBufBytes) + moff;
        uint32_t xm[4][4];
#pragma unroll
        for (int g = 0; g < 4; ++g) ldmatrix_x4_trans(bx0 + g * 512, xm[g]);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
#pragma unroll
          for (int pb = 0; pb < 4; ++pb) xm[g][pb] = bf2_fma(ncs2[pb], xm[g][pb], pa[g][pb]);
          stmatrix_x4_trans(bx0 + g * 512, xm[g]);
        }
        fence_proxy_async_smem();
        __syncwarp();
        RC_TACC(2, tmath);
        if (lane == 0) {
          if (!(prm.ablate & 2)) {
            if (kKB && prm.acc_dx) tma_reduce_add_3d(&map_dx, ebuf + bi * kEpiBufBytes, cs.px, cs.u * 64 + h * 32, cs.bo);
            else tma_store_3d_hint(&map_dx, ebuf + bi * kEpiBufBytes, cs.px, cs.u * 64 + h * 32, cs.bo, pol_first);
            tma_store_commit();
          }
          if (s_req < total) {
            // the box to refill was stored kEpiBufs - kEpiAhead steps ago: that store must have read it
            RC_T0(tsw);
            asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kEpiBufs - kEpiAhead) : "memory");
            RC_TACC(5, tsw);
            request_x();
          }
        }
        cursor_next(cs);
        if (s_req < total) { cursor_next(cr); ++s_req; }
        __syncwarp();
        if (warp == 12 && blk < 8) RC_EV(l, 21 + 2 * blk);      // block drained, its store issued
      }
    }
    if (lane == 0) tma_store_wait_all0();       // shared memory must stay valid until the last bulk store has read it
  }
#ifdef RC_TIMING
  // roles: 0 text producer, 1 MMA issuer, 2 softmax (warp 4), 3 dX epilogue (warp 12), 4 X producer
  if (prm.dbg != nullptr && blockIdx.x < 2 && lane == 0 && (warp <= 1 || warp == 3 || warp == 4 || warp == 12)) {
    wt[0] = clock64() - t_start;
    const int role = warp == 0 ? 0 : (warp == 1 ? 1 : (warp == 4 ? 2 : (warp == 12 ? 3 : 4)));
#pragma unroll
    for (int i = 0; i < 16; ++i) prm.dbg[(blockIdx.x * 5 + role) * 16 + i] = wt[i];
  }
#endif
  tc_fence_before();
  cluster_sync();            // no CTA leaves while its peer may still touch its barriers / shared memory
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_2sm<kTmemCols>(tmem);
  }
}

}  // namespace ts

// launch helper used by rc_infonce_bf16 for backward launches without dText (infonce.cu owns argument checking)
int launch_infonce_ts(const InfoncePairArgs& a, cudaStream_t s) {
  using namespace ts;
  CUtensorMap m_xs, m_t, m_tt, m_xe, m_dx;
  int rcode;
  if ((rcode = make_operand_maps(a, 32, {"ts map_x_s", "ts map_t", "ts map_tt"}, &m_xs, &m_t, &m_tt))) return rcode;
  if ((rcode = make_xmap(&m_xe, a.xsrc, a, a.kb > 0 ? 1 : a.B, 32, 32, "ts map_xe"))) return rcode;
  if ((rcode = make_xmap(&m_dx, a.dx, a, a.B, 32, 32, "ts map_dx"))) return rcode;
  Params prm;
  int grid = 0;
  if ((rcode = fill_tiling(prm, a, &grid))) return rcode;
  prm.k_dev = a.k_dev; prm.log_tau_dev = a.log_tau_dev; prm.k0 = a.k0;
  auto launch = [&](auto kernel) -> int {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
    if (e != cudaSuccess) return fail(RC_ERR_CUDA, "rc_infonce_bf16(ts): smem opt-in: %s", cudaGetErrorString(e));
    kernel<<<grid, kThreads, kSmemBytes, s>>>(m_xs, m_t, m_tt, m_xe, m_dx, prm);
    return check_launch("rc_infonce_bf16(ts)");
  };
  if (a.rep == 4) return launch_kblocked(a) ? launch(infonce_ts_kernel<4, true>) : launch(infonce_ts_kernel<4, false>);
  if (launch_kblocked(a)) return launch(infonce_ts_kernel<1, true>);
  return launch(infonce_ts_kernel<1, false>);
}

}  // namespace rc
