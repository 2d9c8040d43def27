// What the two CTA-pair InfoNCE kernels share: infonce_umma2.cu (SS: both dX operands in shared memory) and
// infonce_ts.cu (TS: the softmax tile is a tensor-memory operand of the dX GEMM).
//
// The two kernels must produce bit-identical dX and lse, so everything that decides a value exists once, here: the
// tiling of the pixels into tile pairs, the operand producers (text and X rings, the relay of X arrivals to the leader
// CTA), the softmax warps' arithmetic (row norms, row max, exp pass, targets, lse and loss, the gradient scales) and the
// host code that builds the shared tensor maps and Params fields.  Each kernel keeps its pipeline, where P goes, where
// the running loss / weight / dlogtau sums live, and its dX epilogue.
//
// Role layout of both kernels (640 threads): warp 0 text TMA, 1 MMA (leader CTA), 2 relay + TMEM alloc, 3 X TMA,
// 4-11 softmax (two warps per TMEM lane quarter: half 0 takes text columns [0, Kp/2), half 1 the rest), 12-19 dX epilogue.
#pragma once
#include "common.cuh"
#include "umma.cuh"
#include "infonce_device.cuh"
#include <float.h>
#include <stdlib.h>

namespace rc {
namespace cta_pair {
using namespace umma;

constexpr int kTilePx = 128;           // pixels per tile (one CTA); a cluster works on tile pairs (2 pj, 2 pj + 1)
constexpr int kStageBytes = 16 * 1024; // one slot of the X and text rings

// The Params fields of both kernels.  Each kernel's Params derives from it.
struct Tiling {
  long long* dbg;           // timing build: per-role wait cycles and the event trace (tools/timing_pair.py, timing_ts.py)
  int ablate;               // bring-up only (RANGECLIP_B200_ABLATE); the bits each kernel reads are listed at its Params
  int B, D, K, Kp;
  int64_t HW;
  int tiles_per_img, n_tiles, n_pairs;
  uint32_t tpi_magic;       // floor(2^32 / tiles_per_img): tile / tiles_per_img as a multiply-high + one correction
  // K-blocked use (more than 256 candidates, e.g. the area-image loss at thousands of objects): the candidates are split
  // into launches of <= 256 rows.  keep_w: a target outside this launch's rows keeps its weight (only the one-hot term is
  // dropped).  lse_in: the row's logsumexp over ALL candidates, from a first round of forward launches; the softmax of
  // this block is then exp(z - lse_in) instead of exp(z - m) / (block sum).
  int keep_w;
  int acc_dx;               // K-blocked backward launches after the first: dX += this block's gradient (TMA reduce-add store)
  const float* lse_in;
  // kb > 0: ALL candidate blocks in one launch.  The "images" of the tile index are the kb blocks of 256 candidate rows:
  // X (one image) is read with image coordinate 0, everything else (y, w, lse, dX, text rows) is indexed by the block.
  // K is then the total number of candidates; lse_in is indexed by the pixel alone.
  int kb;
  const int32_t* y;
  const float* w;
  float inv_tau;
  const float* grad_scale;
  const double* w_sum_in;
  float* lse;
  double* loss_sum;
  double* w_sum;
  double* dlogtau;
};

// ------------------------------------------------------------------------------------------------
// tiling
// ------------------------------------------------------------------------------------------------
// tile / tiles_per_img without the ~20-instruction runtime division (exact for tile < 2^32: the estimate is low by at most 1)
__device__ __forceinline__ int div_tiles(const Tiling& prm, int tile) {
  int q = (int)__umulhi((uint32_t)tile, prm.tpi_magic);
  if (tile - q * prm.tiles_per_img >= prm.tiles_per_img) ++q;
  return q;
}

// tile -> (image, first pixel); tiles past the end map to image index B, which is out of bounds for every
// tensor map (TMA loads return zeros)
__device__ __forceinline__ void tile_coords(const Tiling& prm, int tile, int& b, int& px0) {
  if (tile < prm.n_tiles) {
    b = div_tiles(prm, tile);
    px0 = (tile - b * prm.tiles_per_img) * kTilePx;
  } else {
    b = prm.B;
    px0 = 0;
  }
}

// first candidate row of pair pj's block (kb mode: both tiles of a pair lie in one block, tiles_per_img is even)
template <bool kKB>
__device__ __forceinline__ int text_row0(const Tiling& prm, int pj) {
  return (kKB && prm.kb > 0) ? div_tiles(prm, 2 * pj) * 256 : 0;
}

// K-blocked launches with the row count in device memory (rc_infonce_bf16_dyn_kblock): the valid rows of the launch's
// block, rows [k0, k0 + K) of the contrast set, of which *k_dev are valid in all.  0 or fewer: an empty launch.  The first
// block keeps at least one row, as the one-launch form does (rows past *k_dev are zero pad rows).
__device__ __forceinline__ int block_rows(const int32_t* k_dev, int k0, int K) {
  const int v = min(K, __ldg(k_dev) - k0);
  return k0 == 0 ? max(1, v) : v;
}

// consumer-release barriers live in the leader CTA
__device__ __forceinline__ void arrive_leader(bool leader_cta, uint64_t* bar) {
  if (leader_cta) mbar_arrive(bar);
  else mbar_arrive_remote(map_to_cta(bar, 0));
}
// one arrival for the whole warp: every lane has fenced its own accesses, __syncwarp orders them before lane 0's arrive
__device__ __forceinline__ void arrive_leader_warp(bool leader_cta, uint64_t* bar) {
  __syncwarp();
  if (elect_one()) arrive_leader(leader_cta, bar);
}

// ------------------------------------------------------------------------------------------------
// producers (one thread each, both CTAs)
// ------------------------------------------------------------------------------------------------
// Text chunks [c_begin, c_end) of the S GEMM: this CTA's half (Kp/2 rows from row koff + rank Kp/2) of each 64-channel
// chunk, into the text ring at `ring`.  `it` counts the ring's fills (the dX operand loads share the ring).
template <int kTStages>
__device__ __forceinline__ void load_text_s(const Tiling& prm, const CUtensorMap* map_t, uint8_t* ring, uint64_t* tfull,
                                            uint64_t* tempty, uint32_t& it, int c_begin, int c_end, int koff, uint32_t rank
                                            RC_WT_PARAM) {
  const int Nh = prm.Kp / 2;
  const bool leader_cta = rank == 0;
  for (int c = c_begin; c < c_end; ++c, ++it) {
    const int st = it % kTStages;
    RC_WAIT(mbar_wait, &tempty[st], ((it / kTStages) & 1) ^ 1, 1);
    if ((prm.ablate & 256) && it >= (uint32_t)kTStages) {      // bring-up: no text traffic after the first ring pass (stale operands)
      if (leader_cta) mbar_arrive(&tfull[st]);
      continue;
    }
    if (leader_cta) mbar_arrive_expect_tx(&tfull[st], 2 * Nh * 128);
    tma_load_2d_2sm(ring + st * kStageBytes, map_t, &tfull[st], c * 64, koff + (int)rank * Nh);
  }
}

// The own X chunks [64 d][128 px] of tile `tile` into the X ring at slot 0 of shared memory.  The chunks land on the
// CTA-local xf barriers (the softmax warps read them for the row norms; the relay forwards them to the leader).
// kHint: the loads carry the L2 policy `pol` (TS: evict_last, for the epilogue's re-read of the tile).
template <int kXStages, bool kKB, bool kHint>
__device__ __forceinline__ void load_x_tile(const Tiling& prm, const CUtensorMap* map_x, uint8_t* smem, uint64_t* xf,
                                            uint64_t* xempty, uint32_t& xit, int tile, int n_dchunks, uint64_t pol,
                                            int tag RC_WT_PARAM) {
  int b, px0;
  tile_coords(prm, tile, b, px0);
  for (int c = 0; c < n_dchunks; ++c, ++xit) {
    const int st = xit % kXStages;
    RC_WAIT(mbar_wait, &xempty[st], ((xit / kXStages) & 1) ^ 1, tag);
    uint8_t* sb = smem + st * kStageBytes;
    mbar_arrive_expect_tx(&xf[st], 2 * 8192);
    const int bx = (kKB && prm.kb > 0) ? (b < prm.B ? 0 : 1) : b;      // kb mode: the one image of X (1 = out of bounds)
    if (kHint) {
      tma_load_3d_hint(sb, map_x, &xf[st], px0, c * 64, bx, pol);
      tma_load_3d_hint(sb + 8192, map_x, &xf[st], px0 + 64, c * 64, bx, pol);
    } else {
      tma_load_3d(sb, map_x, &xf[st], px0, c * 64, bx);
      tma_load_3d(sb + 8192, map_x, &xf[st], px0 + 64, c * 64, bx);
    }
  }
}

// relay of one tile's X chunks: "own X chunk has landed" (CTA-local xf) -> the leader's full barrier (both CTAs' halves
// of the S GEMM's A operand must be there before the leader issues).  kTimed: the wait counts in the timing build's wt[tag].
template <int kXStages, bool kTimed>
__device__ __forceinline__ void relay_x_tile(int n_dchunks, uint64_t* xf, uint64_t* xfull, uint32_t& xit, bool leader_cta,
                                             int tag RC_WT_PARAM) {
  for (int c = 0; c < n_dchunks; ++c, ++xit) {
    const int st = xit % kXStages;
    if (kTimed) RC_WAIT(mbar_wait, &xf[st], (xit / kXStages) & 1, tag);
    else mbar_wait(&xf[st], (xit / kXStages) & 1, tag);
    arrive_leader(leader_cta, &xfull[st]);
  }
}

// ------------------------------------------------------------------------------------------------
// softmax warps: thread = (pixel `row` of the own tile == TMEM lane, half of the text columns)
// ------------------------------------------------------------------------------------------------
// R = targets per embedding row: 1 = one pixel per row (y, w are [B*HW]); 4 = every row stands for the four pixels of a
// 2x2 block that share one embedding (decoder.py:113 nearest x2): y, w are [B*HW][4], the loss of the row is
// sum_j w_j (lse - z[y_j]) and dX is the gradient with respect to the shared embedding (the sum over the block).

// Target(s) and weight of the thread's pixel of tile t, read one tile ahead (`live`: t belongs to this cluster).
// ok = 1 for a valid pixel; R = 4: the four targets, 8 bits each (K <= 256); ignored targets are sorted out when w is read.
// In K-blocked launches a relative target outside [0, 256) (ignored, or in another block) aliases to some column of this
// block here.  That is harmless only because the logit it picks up (exp_pass: sy[j]) is used solely under mine[j], which
// gather_targets computes from the full 32-bit target.
template <int R>
__device__ __forceinline__ void load_pixel_scalars(const Tiling& prm, bool live, int t, int row, float& ok, float& w, int& y) {
  ok = 0.f; w = 0.f; y = -1;
  if (live && t < prm.n_tiles) {
    const int tb = div_tiles(prm, t);
    const int tpx = (t - tb * prm.tiles_per_img) * kTilePx + row;
    if (tpx < prm.HW) {
      const int64_t tm = (int64_t)tb * prm.HW + tpx;
      ok = 1.f;
      if (R == 1) {
        y = __ldg(prm.y + tm);
        w = __ldg(prm.w + tm);
      } else {
        const int4 y4 = __ldg(reinterpret_cast<const int4*>(prm.y) + tm);
        y = (y4.x & 255) | ((y4.y & 255) << 8) | ((y4.z & 255) << 16) | ((y4.w & 255) << 24);
      }
    }
  }
}

// Row norm 1/|x_p| (model.py:272 F.normalize) of the tile whose X chunks come next in the X ring, read where they sit
// ([64 d][2 x 64 px], 128-byte swizzle): thread = (8-pixel group ng, row phase nr) = norm_coords(); sums of squares meet
// in shared memory (part_s: [8 softmax warps][128 px]).  Each warp releases every chunk (xempty).  no_reads: bring-up
// ablation.
__device__ __forceinline__ void norm_coords(int& ng, int& nr) {
  const int st_ = threadIdx.x - 128;                           // 0..255
  ng = st_ & 15; nr = st_ >> 4;
}
template <int kXStages>
__device__ __forceinline__ float norm_tile(const uint8_t* smem, uint64_t* xf, uint64_t* xempty, uint32_t& nit, int n_dchunks,
                                           float* part_s, int warp, int lane, int row, int ng, int nr, bool no_reads,
                                           int tag RC_WT_PARAM) {
  float ss[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) ss[j] = 0.f;
  for (int c = 0; c < n_dchunks; ++c, ++nit) {
    const int st = nit % kXStages;
    RC_WAIT(mbar_wait, &xf[st], (nit / kXStages) & 1, tag);
    const uint8_t* base = smem + st * kStageBytes + (ng >> 3) * 8192 + nr * 128;
    const int ch = ng & 7;
#pragma unroll
    for (int rr = 0; rr < (no_reads ? 0 : 4); ++rr) {
      const int rowd = nr + rr * 16;
      const uint4 v = *reinterpret_cast<const uint4*>(base + rr * 2048 + ((ch ^ (rowd & 7)) << 4));
      const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {       // FHFMA.BF16 on the word's halves: no unpack instructions
        ss[2 * j] = sqacc_bf16x2_lo(ss[2 * j], u[j]);
        ss[2 * j + 1] = sqacc_bf16x2_hi(ss[2 * j + 1], u[j]);
      }
    }
    __syncwarp();
    if (elect_one()) mbar_arrive(&xempty[st]);     // (elect.sync: no lane id to re-materialise in this hot loop)
  }
  // fixed-order reduction (bit-reproducible): lane pairs, then the eight warps' partials through shared memory
#pragma unroll
  for (int j = 0; j < 8; ++j) ss[j] += __shfl_xor_sync(0xffffffffu, ss[j], 16);     // lanes l and l^16: same pixels, other rows
  if (lane < 16) {
    float4* dst = reinterpret_cast<float4*>(part_s + (warp - 4) * 128 + ng * 8);
    dst[0] = make_float4(ss[0], ss[1], ss[2], ss[3]);
    dst[1] = make_float4(ss[4], ss[5], ss[6], ss[7]);
  }
  named_bar_sync(5, 256);
  float q = 0.f;
#pragma unroll
  for (int wv = 0; wv < 8; ++wv) q += part_s[wv * 128 + row];
  return 1.f / fmaxf(sqrtf(q), 1e-12f);
}

// The row maximum over the valid columns of both halves (this half's from TMEM at trow, the other's through xch) times
// zl: the exp offset when inv_tau is too large for the fixed bound
__device__ __forceinline__ float row_max(uint32_t trow, int Kt, int cb, int Kh, float* xch, int half, int row, float zl) {
  float mx = -FLT_MAX;
  for (int c = 0; c * 32 < Kh; ++c) {
    const int nvalid = Kt - (cb + c * 32);
    if (nvalid <= 0) break;
    uint32_t r[32];
    tmem_ld_32x32(trow + c * 32, r);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 32; ++i) if (i < nvalid) mx = fmaxf(mx, __uint_as_float(r[i]));
  }
  xch[(0 * 2 + half) * 128 + row] = mx;
  named_bar_sync(3, 256);
  mx = fmaxf(mx, xch[(0 * 2 + (half ^ 1)) * 128 + row]);
  return mx * zl;
}

// The row's exp offset ml (log2 units): the fixed bound, or the row maximum (row_max; every softmax thread takes the same
// branch, it holds a named barrier).  K-blocked rounds with lse_in: the row's logsumexp over ALL candidates, so that
// e = exp(z - lse) is the softmax itself and row_lse sets sum = 1.  (With this block's own maximum as the offset, sum =
// exp(lse - m) overflows ex2.approx to +inf once lse exceeds the block's largest logit by 128 ln 2 = 88.7 nats -- at tau =
// 0.01 a cosine gap of 0.89 -- and the row's target entry of G becomes (e_y - inf) * 0 = NaN.)  Rows past the end of
// the image (zl = 0, weight 0) take offset 0: e = 1, a finite sum.
template <bool kKB>
__device__ __forceinline__ float row_offset(const Tiling& prm, bool valid, int px, int64_t m, bool use_bound, float ml_bound,
                                            uint32_t trow, int Kt, int cb, int Kh, float* xch, int half, int row, float zl) {
  if (kKB && prm.lse_in != nullptr)
    return valid ? __ldg(prm.lse_in + (prm.kb > 0 ? (int64_t)px : m)) * kLog2e : 0.f;
  return use_bound ? ml_bound : row_max(trow, Kt, cb, Kh, xch, half, row, zl);
}

// The exp pass over this half's Kh columns of S (TMEM at trow, 16 columns per step): e = exp(z - m), kept in registers as
// packed bf16 (pk), with sum = sum e and sez = sum e z (up to the scale zs) of the valid columns (k < Kt), and sy[j] = the
// raw logit of target j if it lies in this half.  yi: the target (R = 1) or the four packed targets (R = 4).  R = 4: sy[j]
// may hold an aliased column's logit (load_pixel_scalars); every reader must guard it with mine[j].
// (Measured, not adopted: the scale / sum / e*s arithmetic as packed fp32x2 -- FFMA2 / FADD2, 6 instead of 9 issued
// instructions per two columns -- is 2.7 % slower, 2.57 against 2.50 ms.)
template <int R>
__device__ __forceinline__ void exp_pass(uint32_t trow, int cb, int Kh, int Kt, int yi, float zl, float ml, uint32_t (&pk)[64],
                                         float (&sy)[R], float& sum, float& sez) {
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f, q0 = 0.f, q1 = 0.f, q2 = 0.f, q3 = 0.f;
#pragma unroll
  for (int j = 0; j < R; ++j) sy[j] = 0.f;
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    if (c * 16 < Kh) {
      uint32_t r[16];
      tmem_ld_32x16(trow + c * 16, r);
      tmem_ld_wait();
      const int k0 = cb + c * 16;
      const int nvalid = Kt - k0;
#pragma unroll
      for (int j = 0; j < R; ++j) {                          // target logit(s): once per row, not per column
        const int yrel = (R == 1 ? yi : (int)(((uint32_t)yi >> (8 * j)) & 255u)) - k0;
        if ((unsigned)yrel < 16u) sy[j] = select16(r, yrel);
      }
      if (nvalid >= 16) {
#pragma unroll
        for (int i = 0; i < 16; i += 4) {
          const float a0 = __uint_as_float(r[i]), a1 = __uint_as_float(r[i + 1]);
          const float a2 = __uint_as_float(r[i + 2]), a3 = __uint_as_float(r[i + 3]);
          const float e0 = fast_exp2(fmaf(a0, zl, -ml)), e1 = fast_exp2(fmaf(a1, zl, -ml));
          const float e2 = fast_exp2(fmaf(a2, zl, -ml)), e3 = fast_exp2(fmaf(a3, zl, -ml));
          s0 += e0; s1 += e1; s2 += e2; s3 += e3;
          q0 = fmaf(e0, a0, q0); q1 = fmaf(e1, a1, q1); q2 = fmaf(e2, a2, q2); q3 = fmaf(e3, a3, q3);
          pk[c * 8 + (i >> 1)] = pack_bf16x2(e0, e1);
          pk[c * 8 + (i >> 1) + 1] = pack_bf16x2(e2, e3);
        }
      } else {          // the step that straddles K, or padding columns only
#pragma unroll
        for (int i = 0; i < 16; i += 2) {
          const float a0 = __uint_as_float(r[i]), a1 = __uint_as_float(r[i + 1]);
          const float e0 = (i < nvalid) ? fast_exp2(fmaf(a0, zl, -ml)) : 0.f;
          const float e1 = (i + 1 < nvalid) ? fast_exp2(fmaf(a1, zl, -ml)) : 0.f;
          s0 += e0; s1 += e1;
          q0 = fmaf(e0, a0, q0); q1 = fmaf(e1, a1, q1);
          pk[c * 8 + (i >> 1)] = pack_bf16x2(e0, e1);
        }
      }
    }
  }
  sum = (s0 + s1) + (s2 + s3);
  sez = (q0 + q1) + (q2 + q3);
}

// Targets of the row: y_j, w_j (w_j = 0: ignored), mine[j] = target j lies in this half's columns [cb, cb + Kh),
// wtot = sum_j w_j and tz = sum_j w_j sy[j] over the targets in this half.  R = 1 takes yi / wi from the pixel scalars;
// R = 4 reads the four targets and weights of pixel m if its pixel-scalar flag `ok` is set.  K-blocked launches with
// keep_w (kKB): a target outside this launch's rows (y < 0 included) keeps its weight, so that wtot is the row's weight
// over all blocks; ignored targets then carry w = 0 (rangeclip_b200.h, RC_INFONCE_KEEP_WEIGHT).
template <int R, bool kKB>
__device__ __forceinline__ void gather_targets(const Tiling& prm, int yi, float wi, float ok, int64_t m, int cb, int Kh,
                                               const float (&sy)[R], int (&yj)[R], float (&wj)[R], bool (&mine)[R],
                                               float& wtot, float& tz) {
  if (R == 1) {
    yj[0] = yi; wj[0] = wi;
  } else {
    int4 y4 = make_int4(-1, -1, -1, -1);
    float4 w4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ok != 0.f) {
      y4 = __ldg(reinterpret_cast<const int4*>(prm.y) + m);
      w4 = __ldg(reinterpret_cast<const float4*>(prm.w) + m);
    }
    const int ya[4] = {y4.x, y4.y, y4.z, y4.w};
    const float wa[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
    for (int j = 0; j < R; ++j) { yj[j] = ya[j]; wj[j] = (ya[j] >= 0 || (kKB && prm.keep_w)) ? wa[j] : 0.f; }
  }
  wtot = 0.f; tz = 0.f;
#pragma unroll
  for (int j = 0; j < R; ++j) {
    mine[j] = yj[j] >= cb && yj[j] < cb + Kh;
    wtot += wj[j];
    tz += mine[j] ? wj[j] * sy[j] : 0.f;
  }
}

// The two halves of a row exchange sum, sez and tz through shared memory (xch: [max, sum, sez, sy][2 halves][128]):
// post_sums, then named barrier 2 over the 256 softmax threads, then add_peer_sums
__device__ __forceinline__ void post_sums(float* xch, int half, int row, float sum, float sez, float tz) {
  xch[(1 * 2 + half) * 128 + row] = sum;
  xch[(2 * 2 + half) * 128 + row] = sez;
  xch[(3 * 2 + half) * 128 + row] = tz;
}
__device__ __forceinline__ void add_peer_sums(const float* xch, int half, int row, float& sum, float& sez, float& tz) {
  sum += xch[(1 * 2 + (half ^ 1)) * 128 + row];
  sez += xch[(2 * 2 + (half ^ 1)) * 128 + row];
  tz += xch[(3 * 2 + (half ^ 1)) * 128 + row];
}

// The row's logsumexp (half 0; 0 in half 1), and its loss and weight added to loss / wsum.  K-blocked rounds with
// lse_in: the exp offset was lse_in itself (row_offset), so e is already the softmax over all candidates and sum = 1.
// lse_in is indexed by the embedding row m (R = 4: one lse per shared row) or, in kb mode, by the pixel.
template <bool kKB>
__device__ __forceinline__ float row_lse(const Tiling& prm, bool valid, float ml, int half, float wtot, float tz, float zs,
                                         float& sum, float& loss, float& wsum) {
  if (kKB && prm.lse_in != nullptr && valid) sum = 1.f;
  float lse = 0.f;
  if (half == 0) {
    lse = (ml + __log2f(sum)) * kLn2;
    loss += wtot * lse - tz * zs;
    wsum += wtot;
  }
  return lse;
}

// d loss / d (mean) = coefb = gscale * inv_wsum: grad_scale and 1 / (sum of weights), read once per kernel
__device__ __forceinline__ void grad_scales(const Tiling& prm, float& gscale, float& inv_wsum) {
  const double ws = prm.w_sum_in[0];
  inv_wsum = ws > 0.0 ? (float)(1.0 / ws) : 0.f;
  gscale = prm.grad_scale ? prm.grad_scale[0] : 1.f;
}
// P is stored pre-scaled: G[p][k] = rs_p (e_pk - sum_p [k = y_p]) = d loss / d(xhat_p . that_k) / |x_p|, so the dX
// accumulators need no row scale (and in SS the same tile is the A operand of the dText GEMM, dT = G^T X).  rsv = rs_p / e.
__device__ __forceinline__ float p_scale(float inv_n, float inv_tau, float coef, float inv_sum) {
  return inv_n * inv_tau * coef * inv_sum;
}
// cj: the row's coefficient of the projection term of the normalisation; dx = acc - inv_n^2 cj x, dlogtau -= cj
__device__ __forceinline__ float proj_coef(float coef, float coefb, float sez, float tz, float zs, float inv_sum) {
  return coef * sez * zs * inv_sum - coefb * tz * zs;
}

// G[row][y_j] = rs (e_y - sum * (weight of target y_j) / (weight of the row))  (softmax - onehot), formed before rounding
template <int R>
__device__ __forceinline__ float target_g(int j, const float (&sy)[R], const int (&yj)[R], const float (&wj)[R], float wtot,
                                          float sum, float zl, float ml, float rsv) {
  const float ey = fast_exp2(fmaf(sy[j], zl, -ml));
  if (R == 1) return (ey - sum) * rsv;
  float wk = 0.f;                 // targets of the block that name the same text row
#pragma unroll
  for (int i = 0; i < R; ++i) wk += (yj[i] == yj[j]) ? wj[i] : 0.f;
  return (ey - sum * (wtot > 0.f ? wk / wtot : 0.f)) * rsv;      // rs = rsv carries the block's total weight
}

// the warp's loss, weight and dlogtau sums, added to the float64 totals
template <bool kBwd>
__device__ __forceinline__ void add_sums(const Tiling& prm, int lane, float loss, float wsum, float dlt) {
  loss = warp_sum(loss); wsum = warp_sum(wsum); dlt = warp_sum(dlt);
  if (lane == 0) {
    if (prm.loss_sum) atomicAdd(prm.loss_sum, (double)loss);
    if (prm.w_sum) atomicAdd(prm.w_sum, (double)wsum);
    if (kBwd && prm.dlogtau) atomicAdd(prm.dlogtau, (double)dlt);
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// text rows per launch: Kp = K rounded up to 64; kb mode: blocks of 256
inline int launch_kp(const InfoncePairArgs& a) { return a.kb > 0 ? 256 : (a.K + 63) / 64 * 64; }

// the K-blocked instantiation (kKB) is needed
inline bool launch_kblocked(const InfoncePairArgs& a) {
  return a.keep_w || a.lse_in != nullptr || a.kb > 0 || a.acc_dx;
}

// A [images][D][HW] bf16 tensor (X, dX) with a (box_px, box_d, 1) box
inline int make_xmap(CUtensorMap* m, const void* base, const InfoncePairArgs& a, int images, uint32_t box_px, uint32_t box_d,
                     const char* what) {
  const uint64_t dims[3] = {(uint64_t)a.HW, (uint64_t)a.D, (uint64_t)images};
  const uint64_t str[3] = {2, (uint64_t)a.HW * 2, (uint64_t)a.D * a.HW * 2};
  const uint32_t box[3] = {box_px, box_d, 1};
  return make_tmap_bf16(m, base, 3, dims, str, box, what);
}

// The operand maps of the S GEMM and the dX GEMM's text operand:
//   map_x_s X [B][D][HW], box (64 px, 64 d, 1)
//   map_t   T [Kall][D], box (64 d, Kp/2 rows)
//   map_tt  T^T [D][Kall], box (64 k, tt_box_d d); a forward-only launch (no dX, T^T may be null) gets map_t, unread
// kb > 0: all kb blocks of 256 candidate rows in one launch -- B counts the blocks (virtual images), X has ONE image,
// the text maps span all blocks (row offset = block * 256), dX has one [D][HW] slab per block.
// `what`: the three maps' names in error messages.
inline int make_operand_maps(const InfoncePairArgs& a, uint32_t tt_box_d, const char* const (&what)[3], CUtensorMap* m_xs,
                             CUtensorMap* m_t, CUtensorMap* m_tt) {
  const int Kp = launch_kp(a);
  const int Kall = a.kb > 0 ? a.kb * 256 : Kp;          // rows of the text matrices
  int rcode;
  if ((rcode = make_xmap(m_xs, a.xsrc, a, a.kb > 0 ? 1 : a.B, 64, 64, what[0]))) return rcode;
  const uint64_t tdims[2] = {(uint64_t)a.D, (uint64_t)Kall}, tstr[2] = {2, (uint64_t)a.D * 2};
  const uint32_t tbox[2] = {64, (uint32_t)(Kp / 2)};
  if ((rcode = make_tmap_bf16(m_t, a.t_bf16, 2, tdims, tstr, tbox, what[1]))) return rcode;
  if (a.dx == nullptr) {
    *m_tt = *m_t;
    return RC_OK;
  }
  const uint64_t ttdims[2] = {(uint64_t)Kall, (uint64_t)a.D}, ttstr[2] = {2, (uint64_t)Kall * 2};
  const uint32_t ttbox[2] = {64, tt_box_d};
  return make_tmap_bf16(m_tt, a.tt_bf16, 2, ttdims, ttstr, ttbox, what[2]);
}

// The Tiling fields of a launch and its grid (one cluster of two CTAs per SM pair, at most one per tile pair).  Returns
// RC_OK or the error status.
inline int fill_tiling(Tiling& p, const InfoncePairArgs& a, int* grid) {
  p.dbg = debug_timing_buffer();
  p.ablate = 0;
#ifdef RC_BRINGUP      // ablation switches of the bring-up build (tools/ablate_pair.py, timing_ts.py); the shipped library has no environment knobs
  { const char* ab = getenv("RANGECLIP_B200_ABLATE"); p.ablate = ab ? atoi(ab) : 0; }
#endif
  p.B = a.B; p.D = a.D; p.K = a.K; p.Kp = launch_kp(a); p.HW = a.HW;
  p.tiles_per_img = (int)((a.HW + kTilePx - 1) / kTilePx);
  if ((int64_t)a.B * p.tiles_per_img > 0x3fffffff) return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16: too many tiles");
  p.n_tiles = a.B * p.tiles_per_img;
  p.tpi_magic = p.tiles_per_img == 1 ? 0xffffffffu : (uint32_t)(0x100000000ull / (uint64_t)p.tiles_per_img);
  p.n_pairs = (p.n_tiles + 1) / 2;
  p.y = a.y; p.w = a.w; p.inv_tau = a.inv_tau; p.grad_scale = a.grad_scale;
  p.w_sum_in = a.w_sum_in; p.lse = a.lse; p.loss_sum = a.loss_sum; p.w_sum = a.w_sum; p.dlogtau = a.dlogtau;
  p.keep_w = a.keep_w; p.lse_in = a.lse_in; p.kb = a.kb; p.acc_dx = a.acc_dx;
  if (a.kb > 0 && (p.tiles_per_img & 1)) return fail(RC_ERR_UNSUPPORTED, "rc_infonce_bf16_kblocks: HW must be a multiple of 256");
  int n_clusters = num_sms() / 2;
  if (n_clusters > p.n_pairs) n_clusters = p.n_pairs;
  *grid = 2 * n_clusters;
  return RC_OK;
}

}  // namespace cta_pair
}  // namespace rc
