// K7: top-k text ids per pixel on the tensor cores (evaluation, model.py:164-173).
//
// Replaces `einsum('bdn,cd->bcn')` (a materialised [B, Kr, HW] logit tensor) followed by a sort-based
// `topk(k, dim=1)` and an index gather with one persistent kernel: per 128-pixel tile the bf16 pixel
// rows stay resident in shared memory while the text rows stream past in blocks of 256; the fp32
// logits live only in TMEM (two 256-column buffers, so the scan of block j overlaps the MMA of block
// j+1) and every thread keeps the running top-k of its pixel in registers.
// The ranking by cosine similarity equals the ranking by raw dot product (the per-pixel norm is a
// positive constant), so no normalisation pass over X is needed; ties go to the smaller text index.
#include "common.cuh"
#include "umma.cuh"
#include "eval_metrics.cuh"
#include <float.h>
#include <type_traits>

namespace rc {
using namespace umma;


namespace topk {

constexpr int kThreads = 384;            // warps: 0 TMA, 1 MMA, 2 TMEM alloc, 3 spare, 4-11 top-k scan (two threads per pixel)
constexpr int kTilePx = 128;
constexpr int kXBytes = 128 * 1024;      // X tile [D <= 512][128 px] bf16: D/64 chunks of 16 KB
constexpr int kStages = 3;
constexpr int kStageBytes = 32 * 1024;   // text block chunk [256 k][64 d]
// CTA-pair form (cta_group::2, two tiles per pair): each CTA stages HALF of a text chunk ([128 k][64 d], 16 KB) and the tensor
// cores read the other half from the peer -- half the shared-memory fill and B-operand traffic per SM, which is what paced
// the single-CTA MMA (48 KB of operand reads + 32 KB of fill per chunk against 128 B/clk); the ring gets twice the stages
constexpr int kPairStages = 6;
constexpr int kPairStageBytes = 16 * 1024;
constexpr int kMaxStages = 6;
constexpr int kNB = 256;                 // text rows per block (MMA N)
constexpr int kTmemCols = 512;
constexpr int kMaxK = 8;
constexpr int kMaxChunks = 8;            // D <= 512

struct __align__(8) Bars {
  uint64_t full[kMaxStages], empty[kMaxStages];
  uint64_t x_full[kMaxChunks], x_empty[kMaxChunks];   // per 64-channel chunk of the resident X tile
  uint64_t s_full[2], s_empty[2];
  uint32_t tmem_base, pad;
};
constexpr int kOffRing = kXBytes;
constexpr int kOffThr = kOffRing + kStages * kStageBytes;      // k-th best of every scan thread, read by its partner [256] f32
constexpr int kOffBars = kOffThr + 256 * 4;
static_assert(kPairStages * kPairStageBytes == kStages * kStageBytes, "both forms use the same ring bytes");
constexpr int kSmemBytes = kOffBars + (int)sizeof(Bars);
static_assert(kSmemBytes <= 232448, "shared-memory budget of one SM (227 KB)");

struct Params {
  int B, D, K, k;
  int64_t HW;
  int tiles_per_img, n_tiles, n_blocks;
  const int32_t* k_dev;                  // nullable: number of valid text rows (<= K) read from device memory at kernel start
  const int64_t* index_map;
  int64_t* out;                          // nullable when only the metrics are wanted
  // fused metrics (validate.py:88-139), all nullable together: the histograms of this batch are added to `hist`
  const int64_t* gt;                     // [B*HW] ground-truth ids
  const uint8_t* E;                      // [C][C] equivalence matrix
  const int64_t* cmap;                   // [C] id -> equivalence class
  int C;
  unsigned long long* hist;              // [5][C]
  unsigned long long* counters;          // [3]
  int w;                                 // R = 4: width of the half-resolution rows (HW = h * w); out / gt are [2h][2w]
};

// KT > 0: compile-time k (the insertion network has exactly k stages); KT == 0: run-time k <= kMaxK
template <int KT>
__device__ __forceinline__ void topk_insert(float (&bv)[kMaxK], int (&bi)[kMaxK], int k, float v, int id) {
  // strict '>' keeps the earlier (smaller) index on ties
#pragma unroll
  for (int j = 0; j < (KT > 0 ? KT : kMaxK); ++j) {
    if ((KT > 0 || j < k) && v > bv[j]) {
      const float tv = bv[j]; const int ti = bi[j];
      bv[j] = v; bi[j] = id; v = tv; id = ti;
    }
  }
}
// The same insertion with every comparison taken against the OLD list (depth 3 instead of k dependent compare-and-swap
// stages): v goes to the first position p with v > bv[p], the entries behind it shift down by one, the last one drops.
// A value that does not beat the k-th best changes nothing (all comparisons false), so callers need no guard.  Entries
// that tie exactly keep their order (the serial network above re-orders equal values when it shifts past them).
template <int KT>
__device__ __forceinline__ void topk_insert_par(float (&bv)[kMaxK], int (&bi)[kMaxK], int k, float v, int id) {
  constexpr int N = KT > 0 ? KT : kMaxK;
  bool c[N];
#pragma unroll
  for (int j = 0; j < N; ++j) c[j] = (KT > 0 || j < k) && v > bv[j];
#pragma unroll
  for (int j = N - 1; j >= 1; --j) {       // descending: bv[j - 1] is still the old entry
    const float sv = c[j - 1] ? bv[j - 1] : v;
    const int si = c[j - 1] ? bi[j - 1] : id;
    bv[j] = c[j] ? sv : bv[j];
    bi[j] = c[j] ? si : bi[j];
  }
  bv[0] = c[0] ? v : bv[0];
  bi[0] = c[0] ? id : bi[0];
}
// insertion with an explicit index tie-break (merging lists whose index ranges interleave)
template <int KT>
__device__ __forceinline__ void topk_insert_tie(float (&bv)[kMaxK], int (&bi)[kMaxK], int k, float v, int id) {
#pragma unroll
  for (int j = 0; j < (KT > 0 ? KT : kMaxK); ++j) {
    if ((KT > 0 || j < k) && (v > bv[j] || (v == bv[j] && (unsigned)id < (unsigned)bi[j]))) {
      const float tv = bv[j]; const int ti = bi[j];
      bv[j] = v; bi[j] = id; v = tv; id = ti;
    }
  }
}

// r[i] for a per-thread dynamic i: binary select tree (registers cannot be indexed dynamically)
__device__ __forceinline__ float select32(const uint32_t (&r)[32], int i) {
  float a[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) a[j] = __uint_as_float((i & 1) ? r[2 * j + 1] : r[2 * j]);
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] = (i & 2) ? a[2 * j + 1] : a[2 * j];
#pragma unroll
  for (int j = 0; j < 4; ++j) a[j] = (i & 4) ? a[2 * j + 1] : a[2 * j];
#pragma unroll
  for (int j = 0; j < 2; ++j) a[j] = (i & 8) ? a[2 * j + 1] : a[2 * j];
  return (i & 16) ? a[1] : a[0];
}

// The same select with its first level on the FMA pipe.  Selects, compares and logic operations share the ALU pipe, which
// takes one warp instruction every two cycles per scheduler, and the candidate loop is ~90 % such instructions; the FMA pipe
// next to it is idle.  p in {0.0, 1.0}: r1 * p + r0 * (1 - p) is exact for finite values (one product is the value itself,
// the other a zero), at two FMA-pipe instructions per pair instead of one ALU select.
__device__ __forceinline__ float select32_fma(const uint32_t (&r)[32], int i) {
  float p, q;
  {
    uint32_t pb;
    asm("mad.lo.u32 %0, %1, 0x3f800000, 0;" : "=r"(pb) : "r"((uint32_t)i & 1u));      // IMAD: FMA pipe
    p = __uint_as_float(pb);
    q = 1.0f - p;
  }
  float a[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    float t;
    asm("mul.f32 %0, %1, %2;" : "=f"(t) : "f"(__uint_as_float(r[2 * j])), "f"(q));
    asm("fma.rn.f32 %0, %1, %2, %3;" : "=f"(a[j]) : "f"(__uint_as_float(r[2 * j + 1])), "f"(p), "f"(t));
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) a[j] = (i & 2) ? a[2 * j + 1] : a[2 * j];
#pragma unroll
  for (int j = 0; j < 4; ++j) a[j] = (i & 4) ? a[2 * j + 1] : a[2 * j];
#pragma unroll
  for (int j = 0; j < 2; ++j) a[j] = (i & 8) ? a[2 * j + 1] : a[2 * j];
  return (i & 16) ? a[1] : a[0];
}

// bit 0 of the result = (v > kth), the previous bits move up: one FMA-pipe subtraction (the sign of kth - v) and one funnel
// shift per column instead of a compare, a select and an add on the ALU pipe
__device__ __forceinline__ uint32_t push_gt(uint32_t m, float v, float kth) {
  const uint32_t d = __float_as_uint(kth - v);
  asm("shf.l.wrap.b32 %0, %1, %0, 1;" : "+r"(m) : "r"(d));
  return m;
}

// kPair: launched as clusters of two CTAs (cudaLaunchAttributeClusterDimension); unit of work = a PAIR of tiles, CTA rank r owns
// tile 2 * pair + r; only the leader (rank 0) issues MMAs, which span both SMs (M = 256); completion is multicast to the
// barriers of both CTAs, the scan warps of both CTAs release the S buffer at the leader.
// P = scan threads per pixel (2 or 4): each keeps its own running top-k over 256 / P columns of every block; more lists mean
// more insertions in total but twice the warps to hide the dependent chains behind.
// R = targets per row: 1, or 4 when the rows are the decoder's half-resolution output (SURVEY 8f-1) and every row stands for
// the 2x2 block (2i + a, 2j + b) of the nearest-x2 upsampled map -- the scan is the same, the epilogue writes the ids to the
// block's four pixels and scores each of them against its own full-resolution ground truth.
template <int KT, bool kPair, int P, int R = 1>
__global__ void __launch_bounds__(128 + 128 * P, 1)
eval_topk_umma_kernel(const __grid_constant__ CUtensorMap map_x,    // X [B][D][HW], box (64 px, 64 d, 1)
                      const __grid_constant__ CUtensorMap map_t,    // T [Kp][D], box (64 d, 256 rows; pair: 128 rows), OOB rows = 0
                      const Params prm) {
  extern __shared__ __align__(1024) uint8_t smem[];
  Bars* bars = reinterpret_cast<Bars*>(smem + kOffBars);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_dchunks = prm.D / 64;
  const uint32_t rank = kPair ? cluster_ctarank() : 0u;
  const bool leader_cta = rank == 0;
  constexpr int kRingStages = kPair ? kPairStages : kStages;
  constexpr int kRingBytes = kPair ? kPairStageBytes : kStageBytes;
  // units of work: tiles (single CTA) or tile pairs (CTA pair); a pair's second tile may lie past the end (TMA zero fill)
  const int unit0 = kPair ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int unit_step = kPair ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int n_units = kPair ? (prm.n_tiles + 1) / 2 : prm.n_tiles;
  auto tile_of = [&](int u) -> int { return kPair ? 2 * u + (int)rank : u; };
  // the candidate set may have been built on the device (rc_contrast_build): its size is read here, by every role alike
  const int Kv = prm.k_dev != nullptr ? max(1, min(__ldg(prm.k_dev), prm.K)) : prm.K;
  const int n_blocks = prm.k_dev != nullptr ? (Kv + kNB - 1) / kNB : prm.n_blocks;
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_x); tma_prefetch_desc(&map_t);
    for (int i = 0; i < kMaxStages; ++i) { mbar_init(&bars->full[i], 1); mbar_init(&bars->empty[i], 1); }
    for (int i = 0; i < kMaxChunks; ++i) { mbar_init(&bars->x_full[i], 1); mbar_init(&bars->x_empty[i], 1); }
    // S buffers: released by ONE arrival per scan warp (of both CTAs in the pair form)
    for (int i = 0; i < 2; ++i) { mbar_init(&bars->s_full[i], 1); mbar_init(&bars->s_empty[i], (kPair ? 2 : 1) * 4 * P); }
    fence_barrier_init();
  }
  if (warp == 2) {
    if (kPair) tmem_alloc_2sm<kTmemCols>(&bars->tmem_base);
    else tmem_alloc<kTmemCols>(&bars->tmem_base);
  }
  tc_fence_before();
  if (kPair) cluster_sync();      // both CTAs' barriers are initialised before any remote arrive / 2-SM TMA credit
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem = bars->tmem_base;
  const uint32_t idesc = make_idesc_bf16(kPair ? 256 : 128, kNB, /*A MN-major*/ 1, /*B K-major*/ 0);

  if (warp < 4) {
  // 640 threads x 96 registers at launch (P = 4): the four control warps give registers to the sixteen scan warps
  if (P == 4) asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
  if (warp == 0 && lane == 0) {
    // =============================== TMA producer ===============================
    // X chunk c of the next tile is refilled as soon as the last text block of this tile has consumed it, so the
    // tile transition overlaps with the tail of the tensor work.
    uint32_t it = 0, lt = 0;
    for (int u = unit0; u < n_units; u += unit_step, ++lt) {
      const int tile = tile_of(u);
      const bool tile_ok = tile < prm.n_tiles;
      const int b = tile_ok ? tile / prm.tiles_per_img : prm.B;           // image index B: out of bounds, TMA fills zeros
      const int px0 = tile_ok ? (tile - b * prm.tiles_per_img) * kTilePx : 0;
      for (int nb = 0; nb < n_blocks; ++nb)
        for (int c = 0; c < n_dchunks; ++c, ++it) {
          if (nb == 0) {
            mbar_wait(&bars->x_empty[c], (lt & 1) ^ 1, 1);
            if (kPair) {          // both CTAs' bytes are credited to the leader's barrier
              if (leader_cta) mbar_arrive_expect_tx(&bars->x_full[c], 2 * 16384);
              tma_load_3d_2sm(smem + c * 16384, &map_x, &bars->x_full[c], px0, c * 64, b);
              tma_load_3d_2sm(smem + c * 16384 + 8192, &map_x, &bars->x_full[c], px0 + 64, c * 64, b);
            } else {
              mbar_arrive_expect_tx(&bars->x_full[c], 16384);
              tma_load_3d(smem + c * 16384, &map_x, &bars->x_full[c], px0, c * 64, b);
              tma_load_3d(smem + c * 16384 + 8192, &map_x, &bars->x_full[c], px0 + 64, c * 64, b);
            }
          }
          const int st = it % kRingStages;
          mbar_wait(&bars->empty[st], ((it / kRingStages) & 1) ^ 1, 2);
          if (kPair) {            // own half (128 rows) of the block's chunk
            if (leader_cta) mbar_arrive_expect_tx(&bars->full[st], 2 * kRingBytes);
            tma_load_2d_2sm(smem + kOffRing + st * kRingBytes, &map_t, &bars->full[st], c * 64, nb * kNB + (int)rank * (kNB / 2));
          } else {
            mbar_arrive_expect_tx(&bars->full[st], kRingBytes);
            tma_load_2d(smem + kOffRing + st * kRingBytes, &map_t, &bars->full[st], c * 64, nb * kNB);
          }
        }
    }
  } else if (warp == 1 && leader_cta) {
    // =============================== MMA issuer (leader CTA in the pair form) ================================
    // whole warp converged (addresses / descriptors in uniform registers), one elected lane issues
    uint32_t it = 0, lt = 0, nbc = 0;
    const uint32_t smem_base = smem_u32(smem);
    const uint64_t dsc_x = desc_mnmajor_sw128(0, 8192) + (smem_base >> 4);
    const uint64_t dsc_t = desc_kmajor_sw128(0) + ((smem_base + kOffRing) >> 4);
    for (int u = unit0; u < n_units; u += unit_step, ++lt) {
      for (int nb = 0; nb < n_blocks; ++nb, ++nbc) {
        const int sbuf = nbc & 1;
        mbar_wait(&bars->s_empty[sbuf], ((nbc >> 1) & 1) ^ 1, 4);
        tc_fence_after();
        const bool last = nb + 1 == n_blocks;
        for (int c = 0; c < n_dchunks; ++c, ++it) {
          const int st = it % kRingStages;
          if (nb == 0) mbar_wait(&bars->x_full[c], lt & 1, 3);
          mbar_wait(&bars->full[st], (it / kRingStages) & 1, 5);
          tc_fence_after();
          const uint64_t xa = dsc_x + ((c * 16384) >> 4);
          const uint64_t tb = dsc_t + ((st * kRingBytes) >> 4);
          if (elect_one()) {
            if (kPair) {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)
                mma_bf16_ss_2sm(tmem + sbuf * kNB, xa + ((ks * 2048) >> 4), tb + ((ks * 32) >> 4), idesc, (c | ks) != 0);
              mma_commit_2sm(&bars->empty[st]);
              if (last) mma_commit_2sm(&bars->x_empty[c]);
            } else {
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)
                mma_bf16_ss(tmem + sbuf * kNB, xa + ((ks * 2048) >> 4), tb + ((ks * 32) >> 4), idesc, (c | ks) != 0);
              mma_commit(&bars->empty[st]);
              if (last) mma_commit(&bars->x_empty[c]);       // this X chunk has been read for the last time
            }
          }
          __syncwarp();
        }
        if (elect_one()) {
          if (kPair) mma_commit_2sm(&bars->s_full[sbuf]);
          else mma_commit(&bars->s_full[sbuf]);
        }
        __syncwarp();
      }
    }
  }
  } else {
    if (P == 4) asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
    // =============================== top-k scan ================================
    // Two warps per TMEM lane quarter: half 0 (warps 4-7) scans text columns [0,128) of every 256-row block, half 1
    // (warps 8-11) columns [128,256); each thread keeps a running top-k, the two lists of a pixel are merged at the
    // end of the tile (half 1 parks its list in its own, already scanned TMEM columns).
    const int half = (warp - 4) >> 2;          // which 256 / P columns of a block this thread scans ("half": P = 2)
    constexpr int kCols = kNB / P;             // columns per thread per block
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const uint32_t trow = tmem + ((uint32_t)(quarter * 32) << 16) + half * kCols;
    uint32_t nbc = 0;
    unsigned int m_c1 = 0, m_ck = 0, m_tot = 0;      // fused metrics: per-thread counters
    // The two scan threads of a pixel publish their running k-th best; the partner's value (possibly stale -- every earlier
    // value is still a valid bound) tightens the candidate filter: a value below the k-th best of EITHER column half cannot
    // be among the pixel's top k.  Values EQUAL to the partner's bound stay candidates (the index tie-break is the merge's).
    volatile float* thr_mine = reinterpret_cast<volatile float*>(smem + kOffThr) + (threadIdx.x - 128);
    volatile float* thr_peer = reinterpret_cast<volatile float*>(smem + kOffThr) + ((threadIdx.x - 128) ^ 128);
    *thr_mine = -FLT_MAX;
    named_bar_sync(4 + quarter, 64);
    for (int u = unit0; u < n_units; u += unit_step) {
      const int tile = tile_of(u);
      const bool tile_ok = tile < prm.n_tiles;         // (a pair's second tile past the end: scanned, never written)
      const int b = tile_ok ? tile / prm.tiles_per_img : 0;
      const int px = tile_ok ? (tile - b * prm.tiles_per_img) * kTilePx + row : (int)min((int64_t)0x7fffffff, prm.HW);
      float bv[kMaxK];
      int bi[kMaxK];
#pragma unroll
      for (int j = 0; j < kMaxK; ++j) { bv[j] = -FLT_MAX; bi[j] = -1; }
      float kth = -FLT_MAX;              // current k-th best: cheap reject before the insertion network
      for (int nb = 0; nb < n_blocks; ++nb, ++nbc) {
        const int sbuf = nbc & 1;
        mbar_wait(&bars->s_full[sbuf], (nbc >> 1) & 1, 6);
        tc_fence_after();
        // The TMEM load of the NEXT 32 columns is in flight while this chunk is scanned (two register buffers): with two
        // scan warps per scheduler the exposed tcgen05.ld latency of every chunk was a fifth of the scan time.
        const int kbase = nb * kNB + half * kCols;
        const int n_chunks = min(kCols / 32, max(0, (Kv - kbase + 31) >> 5));
        auto scan_chunk = [&](const uint32_t (&r)[32], int c) {
          const int k0 = kbase + c * 32;
          const int nvalid = Kv - k0;
          if (KT == 1) {
            // arg-max: a branch-free running maximum with static register indices (3 instructions per column) is
            // cheaper than the bitmask + candidate loop at every position of the scan
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const float v = __uint_as_float(r[i]);
              const bool better = (i < nvalid) && (v > bv[0]);       // strict: the smaller index wins ties
              bv[0] = better ? v : bv[0];
              bi[0] = better ? k0 + i : bi[0];
            }
            return;
          }
          if (nb == 0 && c == 0) {
            // The first 32 columns of a tile all beat the empty list: the candidate loop below would run 32 rounds of
            // dynamic register selection (a third of all its rounds in a K = 1024 scan).  Insert them with static
            // register indices instead: no bit scan, no select tree, no branch.
            if (nvalid >= 32) {            // the common case without 32 guards
#pragma unroll
              for (int i = 0; i < 32; ++i) topk_insert_par<KT>(bv, bi, prm.k, __uint_as_float(r[i]), k0 + i);
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i)
                if (i < nvalid) topk_insert_par<KT>(bv, bi, prm.k, __uint_as_float(r[i]), k0 + i);
            }
            if (KT > 0) {
              kth = bv[KT - 1];
            } else {
              kth = bv[0];
#pragma unroll
              for (int j = 1; j < kMaxK; ++j) if (j < prm.k) kth = bv[j];
            }
            if (P == 2) *thr_mine = kth;
            return;
          }
          // Per thread only ~k ln(K/k) values ever enter the top-k, but with 32 pixels per warp some lane qualifies at
          // almost every column.  So: a branch-free candidate bitmask first (four independent chains), then a short
          // per-thread loop over the set bits -- the warp iterates max-over-lanes(#candidates), not once per column.
          float kf = kth;
          if (P == 2) {
            const float pk = *thr_peer;
            if (pk > kth) {              // v >= pk  <=>  v > the float just below pk
              const uint32_t ub = __float_as_uint(pk);
              kf = __uint_as_float(pk > 0.f ? ub - 1u : (pk < 0.f ? ub + 1u : 0x80000001u));
            }
          }
          uint32_t m0 = 0, m1 = 0, m2 = 0, m3 = 0;
#pragma unroll
          for (int i = 7; i >= 0; --i) {            // last pushed = lowest bit: column 8 q + i ends at bit i of chain q
            m0 = push_gt(m0, __uint_as_float(r[i]), kf);
            m1 = push_gt(m1, __uint_as_float(r[8 + i]), kf);
            m2 = push_gt(m2, __uint_as_float(r[16 + i]), kf);
            m3 = push_gt(m3, __uint_as_float(r[24 + i]), kf);
          }
          uint32_t mask = __byte_perm(__byte_perm(m0, m1, 0x0040), __byte_perm(m2, m3, 0x0040), 0x5410);
          if (nvalid < 32) mask &= (1u << nvalid) - 1u;
          if (mask) {
            // Software-pipelined candidate loop: the value of the NEXT candidate is selected (31-instruction tree) while the
            // current one goes through the insertion -- two independent instruction streams per round instead of one
            // serial chain (the scan warps are two per scheduler: their speed is the length of the dependent chain).
            int i = __ffs(mask) - 1;             // ascending column order: the earlier index wins ties
            mask &= mask - 1;
            float v = select32_fma(r, i);
            for (;;) {
              const uint32_t more = mask;
              const int i2 = (__ffs(mask) - 1) & 31;
              mask &= mask - 1;
              const float v2 = select32_fma(r, i2);
              topk_insert_par<KT>(bv, bi, prm.k, v, k0 + i);       // a no-op when v no longer beats the k-th best
              if (!more) break;
              i = i2; v = v2;
            }
            if (KT > 0) {
              kth = bv[KT - 1];
            } else {
              kth = bv[0];
#pragma unroll
              for (int j = 1; j < kMaxK; ++j) if (j < prm.k) kth = bv[j];
            }
            if (P == 2) *thr_mine = kth;
          }
        };
        if (P == 2) {
          uint32_t ra[32], rb[32];
          if (n_chunks > 0) tmem_ld_32x32(trow + sbuf * kNB, ra);
#pragma unroll 1
          for (int c = 0; c < n_chunks; c += 2) {
            tmem_ld_wait32(ra);
            if (c + 1 < n_chunks) tmem_ld_32x32(trow + sbuf * kNB + (c + 1) * 32, rb);
            scan_chunk(ra, c);
            if (c + 1 < n_chunks) {
              tmem_ld_wait32(rb);
              if (c + 2 < n_chunks) tmem_ld_32x32(trow + sbuf * kNB + (c + 2) * 32, ra);
              scan_chunk(rb, c + 1);
            }
          }
        } else {
#pragma unroll 1
          for (int c = 0; c < n_chunks; ++c) {
            uint32_t r[32];
            tmem_ld_32x32(trow + sbuf * kNB + c * 32, r);
            tmem_ld_wait();
            scan_chunk(r, c);
          }
        }
        if (nb + 1 == n_blocks) {
          // merge the P lists of a pixel: parts 1.. park theirs in 16 TMEM columns of their own, already scanned range of
          // this buffer; part 0 folds them into its list (explicit index tie-break: the ranges interleave across blocks)
          const uint32_t tq = tmem + ((uint32_t)(quarter * 32) << 16) + sbuf * kNB;
          *thr_mine = -FLT_MAX;            // the bound belongs to this tile's pixel: reset before the barrier both partners pass
          if (half != 0) {
            uint32_t pkd[16];
#pragma unroll
            for (int j = 0; j < kMaxK; ++j) { pkd[j] = __float_as_uint(bv[j]); pkd[8 + j] = (uint32_t)bi[j]; }
            tmem_st_32x16(tq + half * kCols, pkd);
            tmem_st_wait();
            tc_fence_before();
            named_bar_sync(4 + quarter, 32 * P);
          } else {
            named_bar_sync(4 + quarter, 32 * P);
            tc_fence_after();
#pragma unroll 1
            for (int part = 1; part < P; ++part) {
              uint32_t pkd[16];
              tmem_ld_32x16(tq + part * kCols, pkd);
              tmem_ld_wait();
#pragma unroll
              for (int j = 0; j < kMaxK; ++j)
                if (j < prm.k && (int)pkd[8 + j] >= 0) topk_insert_tie<KT>(bv, bi, prm.k, __uint_as_float(pkd[j]), (int)pkd[8 + j]);
            }
          }
        }
        tc_fence_before();
        __syncwarp();                                   // one release per warp (at the leader in the pair form)
        if (lane == 0) {
          if (leader_cta) mbar_arrive(&bars->s_empty[sbuf]);
          else mbar_arrive_remote(map_to_cta(&bars->s_empty[sbuf], 0));
        }
      }
      if (half == 0) {               // warps 4-7: lane = pixel, 32 consecutive pixels of one image per warp
        const bool inb = px < prm.HW;
        int64_t ids[kMaxK];
#pragma unroll
        for (int j = 0; j < kMaxK; ++j) ids[j] = (inb && j < prm.k && bi[j] >= 0) ? __ldg(prm.index_map + bi[j]) : -1;
        auto id_of = [&](int j) {
          int64_t v = ids[0];
#pragma unroll
          for (int q = 1; q < kMaxK; ++q) v = (j == q) ? ids[q] : v;
          return v;
        };
        // Fused metrics: the pixel's top-k ids never leave the registers on their way into the five class histograms
        // (warp-aggregated atomics: one per distinct class per warp); same per-pixel function as rc_eval_hist.
        auto count = [&](int64_t g) {
          PixelMetric m;
          m.ok = false; m.ge = 0; m.p1 = 0; m.orc = 0; m.top1_same = false; m.orc_same = false; m.any_eq1 = false; m.any_eqk = false;
          if (inb) m = pixel_metric(g, prm.k, id_of, prm.E, prm.cmap, prm.C);
          if (m.ok) { m_c1 += m.any_eq1 ? 1u : 0u; m_ck += m.any_eqk ? 1u : 0u; m_tot += 1u; }
          warp_agg_add(prm.hist + 0 * (int64_t)prm.C, m.ge, m.ok);
          warp_agg_add(prm.hist + 1 * (int64_t)prm.C, m.p1, m.ok);
          warp_agg_add(prm.hist + 2 * (int64_t)prm.C, m.ge, m.ok && m.top1_same);
          warp_agg_add(prm.hist + 3 * (int64_t)prm.C, m.orc, m.ok);
          warp_agg_add(prm.hist + 4 * (int64_t)prm.C, m.ge, m.ok && m.orc_same);
        };
        if (R == 1) {
          if (inb && prm.out != nullptr) {
#pragma unroll
            for (int j = 0; j < kMaxK; ++j)
              if (j < prm.k) prm.out[((int64_t)b * prm.k + j) * prm.HW + px] = ids[j];
          }
          if (prm.hist != nullptr) count(inb ? __ldg(prm.gt + (int64_t)b * prm.HW + px) : 0);
        } else {
          // row (i, j) = full-resolution pixels (2i + a, 2j + c) of a [2h][2w] map: per image row a the two pixels are adjacent
          // from an even index, so each id is one 16-byte store per image row and their gt words one 16-byte load
          const int i = px / prm.w, jx = px - i * prm.w;
          const int64_t W2 = 2 * (int64_t)prm.w, HW4 = 4 * prm.HW;
          const int64_t p00 = 2 * (int64_t)i * W2 + 2 * jx;
          if (inb && prm.out != nullptr) {
#pragma unroll
            for (int j = 0; j < kMaxK; ++j)
              if (j < prm.k) {
                longlong2* o = reinterpret_cast<longlong2*>(prm.out + ((int64_t)b * prm.k + j) * HW4 + p00);
                const longlong2 v = make_longlong2(ids[j], ids[j]);
                o[0] = v;
                o[W2 / 2] = v;
              }
          }
          if (prm.hist != nullptr) {
            longlong2 g0 = make_longlong2(0, 0), g1 = g0;
            if (inb) {
              const longlong2* gp = reinterpret_cast<const longlong2*>(prm.gt + (int64_t)b * HW4 + p00);
              g0 = __ldg(gp);
              g1 = __ldg(gp + W2 / 2);
            }
            // the four pixels share the id list and are counted one by one, exactly as the upsampled launch counts them
#pragma unroll 1
            for (int q = 0; q < 4; ++q) count(q == 0 ? g0.x : q == 1 ? g0.y : q == 2 ? g1.x : g1.y);
          }
        }
      }
    }
    if (half == 0 && prm.hist != nullptr) {
      for (int o = 16; o > 0; o >>= 1) {
        m_c1 += __shfl_xor_sync(0xffffffffu, m_c1, o);
        m_ck += __shfl_xor_sync(0xffffffffu, m_ck, o);
        m_tot += __shfl_xor_sync(0xffffffffu, m_tot, o);
      }
      if (lane == 0) {
        if (m_c1) atomicAdd(&prm.counters[0], (unsigned long long)m_c1);
        if (m_ck) atomicAdd(&prm.counters[1], (unsigned long long)m_ck);
        if (m_tot) atomicAdd(&prm.counters[2], (unsigned long long)m_tot);
      }
    }
  }
  tc_fence_before();
  if (kPair) cluster_sync();      // no CTA leaves while its peer may still touch its barriers / shared memory
  else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    if (kPair) tmem_dealloc_2sm<kTmemCols>(tmem);
    else tmem_dealloc<kTmemCols>(tmem);
  }
}

}  // namespace topk
}  // namespace rc

static int eval_topk_bf16_impl(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW, const void* t_bf16, int K,
                               const int64_t* index_map, int k, int64_t* out, const int64_t* gt, const uint8_t* E,
                               const int64_t* cmap, int C, int64_t* hist, int64_t* counters, void* workspace,
                               int64_t workspace_bytes, void* stream, const char* who, const int32_t* k_dev = nullptr,
                               int rep_w = 0) {
  // rep_w = 0: one target per row (x is [B][D][HW], out / gt [B][HW]); rep_w = w > 0: x holds the half-resolution rows
  // [B][D][h*w] (HW = h*w) and out / gt are the full-resolution [B][2h][2w] maps (four targets per row)
  using namespace rc;
  RC_REQUIRE(x && t_bf16 && index_map && (out || hist), "%s: null pointer", who);
  RC_REQUIRE(B >= 0 && HW >= 0 && K >= 1 && k >= 1 && k <= topk::kMaxK && k <= K, "%s: bad shape (k=%d K=%d)", who, k, K);
  if (hist != nullptr) RC_REQUIRE(gt && E && cmap && counters && C >= 1, "%s: the fused metrics need gt, E, cmap, counters and C >= 1", who);
  if (D < 64 || D > 512 || D % 64 != 0) return fail(RC_ERR_UNSUPPORTED, "%s: D=%d must be a multiple of 64 and <= 512", who, D);
  if (HW % 8 != 0) return fail(RC_ERR_UNSUPPORTED, "%s: HW=%lld must be a multiple of 8", who, (long long)HW);
  if (rep_w > 0)             // 16-byte stores of the ids / loads of the gt words (pixel pairs from an even index)
    RC_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0 && (reinterpret_cast<uintptr_t>(gt) & 15) == 0,
               "%s: out and gt must be 16-byte aligned", who);
  RC_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(t_bf16) & 15) == 0,
             "%s: x and t must be 16-byte aligned", who);
  if (B == 0 || HW == 0) return RC_OK;
  int rcode = check_sm100(who);
  if (rcode) return rcode;
  cudaStream_t s = (cudaStream_t)stream;
  const void* xsrc = x;
  if (x_dtype == RC_F32) {
    const int64_t M = (int64_t)B * HW;
    RC_REQUIRE(workspace && workspace_bytes >= rc_infonce_workspace_bytes(B, D, HW, K, RC_F32), "%s: workspace too small for the bf16 copy", who);
    uint8_t* ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
    float* inv_norm = reinterpret_cast<float*>(ws);
    __nv_bfloat16* xb = reinterpret_cast<__nv_bfloat16*>(ws + ((M * 4 + 255) / 256) * 256);
    if ((rcode = launch_rownorm_f32((const float*)x, B, D, HW, xb, inv_norm, s))) return rcode;
    xsrc = xb;
  }
  const int Kp = (K + 63) / 64 * 64;
  CUtensorMap m_x, m_t;
  {
    const uint64_t dims[3] = {(uint64_t)HW, (uint64_t)D, (uint64_t)B};
    const uint64_t str[3] = {2, (uint64_t)HW * 2, (uint64_t)D * HW * 2};
    const uint32_t box[3] = {64, 64, 1};
    if ((rcode = make_tmap_bf16(&m_x, xsrc, 3, dims, str, box, "topk map_x"))) return rcode;
    const uint64_t tdims[2] = {(uint64_t)D, (uint64_t)Kp}, tstr[2] = {2, (uint64_t)D * 2};
    const uint32_t tbox[2] = {64, (uint32_t)topk::kNB};
    if ((rcode = make_tmap_bf16(&m_t, t_bf16, 2, tdims, tstr, tbox, "topk map_t"))) return rcode;
  }
  topk::Params prm;
  prm.B = B; prm.D = D; prm.K = K; prm.k = k; prm.HW = HW;
  prm.tiles_per_img = (int)((HW + topk::kTilePx - 1) / topk::kTilePx);
  if ((int64_t)B * prm.tiles_per_img > 0x7fffffff) return fail(RC_ERR_UNSUPPORTED, "%s: too many tiles", who);
  prm.n_tiles = B * prm.tiles_per_img;
  prm.n_blocks = (K + topk::kNB - 1) / topk::kNB;
  prm.index_map = index_map; prm.out = out; prm.k_dev = k_dev;
  prm.gt = gt; prm.E = E; prm.cmap = cmap; prm.C = C;
  prm.hist = reinterpret_cast<unsigned long long*>(hist); prm.counters = reinterpret_cast<unsigned long long*>(counters);
  prm.w = rep_w;
  // CTA pairs (two tiles per cluster, text chunks shared between the two SMs) whenever there is more than one tile
  const bool pair = prm.n_tiles >= 2 && (prm.n_blocks >= 2 || k == 1);       // one text block per tile: nothing to share, the coupling costs 5 %
  CUtensorMap m_tp = m_t;
  if (pair) {
    const uint64_t tdims[2] = {(uint64_t)D, (uint64_t)Kp}, tstr[2] = {2, (uint64_t)D * 2};
    const uint32_t tbox[2] = {64, (uint32_t)(topk::kNB / 2)};
    if ((rcode = make_tmap_bf16(&m_tp, t_bf16, 2, tdims, tstr, tbox, "topk map_t (pair)"))) return rcode;
  }
  auto launch = [&](auto kernel, bool is_pair, int threads) -> int {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, topk::kSmemBytes);
    if (e != cudaSuccess) return fail(RC_ERR_CUDA, "%s: smem opt-in: %s", who, cudaGetErrorString(e));
    if (!is_pair) {
      const int grid = prm.n_tiles < num_sms() ? prm.n_tiles : num_sms();
      kernel<<<grid, threads, topk::kSmemBytes, s>>>(m_x, m_t, prm);
      return check_launch(who);
    }
    const int n_pairs = (prm.n_tiles + 1) / 2;
    int n_clusters = num_sms() / 2;
    if (n_clusters > n_pairs) n_clusters = n_pairs;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * n_clusters);
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = topk::kSmemBytes;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    e = cudaLaunchKernelEx(&cfg, kernel, m_x, m_tp, prm);
    if (e != cudaSuccess) return fail(RC_ERR_CUDA, "%s: cluster launch: %s", who, cudaGetErrorString(e));
    return check_launch(who);
  };
  // the two k the reference evaluates with (validate.py: top-1 and top-5) get fixed-size insertion networks
  // Two scan threads per pixel.  Measured, not adopted (P = 4, 640 threads, setmaxnreg 40 / 104): four lists per pixel mean 23 %
  // more insertions and the scan is close to its instruction-throughput bound (ALU + FMA pipe at one warp instruction per two
  // cycles each): K = 1024 top-5 1041 against 1147 Mpix/s, K = 256 2258 against 2764.
  auto dispatch = [&](auto r) -> int {
    constexpr int R = decltype(r)::value;
    if (pair) {
      if (k == 1) return launch(topk::eval_topk_umma_kernel<1, true, 2, R>, true, 384);
      if (k == 5) return launch(topk::eval_topk_umma_kernel<5, true, 2, R>, true, 384);
      return launch(topk::eval_topk_umma_kernel<0, true, 2, R>, true, 384);
    }
    if (k == 1) return launch(topk::eval_topk_umma_kernel<1, false, 2, R>, false, 384);
    if (k == 5) return launch(topk::eval_topk_umma_kernel<5, false, 2, R>, false, 384);
    return launch(topk::eval_topk_umma_kernel<0, false, 2, R>, false, 384);
  };
  return rep_w > 0 ? dispatch(std::integral_constant<int, 4>()) : dispatch(std::integral_constant<int, 1>());
}

extern "C" int rc_eval_topk_bf16(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW, const void* t_bf16, int K,
                                 const int64_t* index_map, int k, int64_t* out, void* workspace, int64_t workspace_bytes,
                                 void* stream) {
  RC_REQUIRE(out, "rc_eval_topk_bf16: null pointer");
  return eval_topk_bf16_impl(x, x_dtype, B, D, HW, t_bf16, K, index_map, k, out, nullptr, nullptr, nullptr, 0, nullptr, nullptr,
                             workspace, workspace_bytes, stream, "rc_eval_topk_bf16");
}

extern "C" int rc_eval_topk_hist_bf16(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW, const void* t_bf16, int K,
                                      const int64_t* index_map, int k, int64_t* out, const int64_t* gt, const uint8_t* E,
                                      const int64_t* cmap, int C, int64_t* hist, int64_t* counters, void* workspace,
                                      int64_t workspace_bytes, void* stream) {
  RC_REQUIRE(hist, "rc_eval_topk_hist_bf16: null pointer");
  return eval_topk_bf16_impl(x, x_dtype, B, D, HW, t_bf16, K, index_map, k, out, gt, E, cmap, C, hist, counters, workspace,
                             workspace_bytes, stream, "rc_eval_topk_hist_bf16");
}

/* Same with the number of valid text rows read from device memory (a candidate set built by rc_contrast_build: K is the row
 * count the launch is shaped for, rows past *k_dev are pads); out and hist are both optional, at least one must be given. */
extern "C" int rc_eval_topk_dyn_bf16(const void* x, rc_dtype x_dtype, int B, int D, int64_t HW, const void* t_bf16, int K,
                                     const int32_t* k_dev, const int64_t* index_map, int k, int64_t* out, const int64_t* gt,
                                     const uint8_t* E, const int64_t* cmap, int C, int64_t* hist, int64_t* counters,
                                     void* workspace, int64_t workspace_bytes, void* stream) {
  RC_REQUIRE(k_dev != nullptr, "rc_eval_topk_dyn_bf16: k_dev is required");
  return eval_topk_bf16_impl(x, x_dtype, B, D, HW, t_bf16, K, index_map, k, out, gt, E, cmap, C, hist, counters, workspace,
                             workspace_bytes, stream, "rc_eval_topk_dyn_bf16", k_dev);
}

/* The same on the decoder's half-resolution rows x [B][D][h*w] (the output_conv result): row (i, j) stands for the 2x2 block
 * (2i + a, 2j + b) of the nearest-x2 upsampled map, whose four pixels have the same top-k; out and gt are full resolution. */
extern "C" int rc_eval_topk_bf16_rep4(const void* x, rc_dtype x_dtype, int B, int D, int h, int w, const void* t_bf16, int K,
                                      const int32_t* k_dev, const int64_t* index_map, int k, int64_t* out, const int64_t* gt,
                                      const uint8_t* E, const int64_t* cmap, int C, int64_t* hist, int64_t* counters,
                                      void* workspace, int64_t workspace_bytes, void* stream) {
  RC_REQUIRE(x && t_bf16 && index_map && (out || hist), "rc_eval_topk_bf16_rep4: null pointer");
  RC_REQUIRE(h >= 1 && w >= 1, "rc_eval_topk_bf16_rep4: bad shape (h=%d w=%d)", h, w);
  return eval_topk_bf16_impl(x, x_dtype, B, D, (int64_t)h * w, t_bf16, K, index_map, k, out, gt, E, cmap, C, hist, counters,
                             workspace, workspace_bytes, stream, "rc_eval_topk_bf16_rep4", k_dev, w);
}
