// Blackwell (sm_100a) building blocks written as inline PTX: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 MMA / TMEM allocation / TMEM loads, shared-memory and instruction descriptors.
// No CUTLASS dependency; descriptor bit layouts follow the PTX ISA tables (the same ones
// cute/arch/mma_sm100_desc.hpp encodes).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace rc {
namespace umma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

// ---- mbarrier ---------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_n(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// try_wait suspends the thread in hardware until the phase completes or the time hint expires; with the default
// (short) limit a waiting warp comes back every ~100 cycles and its polling loop steals issue slots from the
// warps that share its scheduler.
constexpr uint32_t kSuspendHintNs = 200000u;
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(kSuspendHintNs)
      : "memory");
  return ok != 0;
}
// Bring-up builds (-DRC_BRINGUP) bound every wait: a protocol bug must surface as a trapped kernel (CUDA error), never as a
// hung GPU.  The shipped build spins on try_wait alone: the clock reads and the timeout branch are ~15 instructions per
// wait in loops that are issue-bound.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int tag) {
#ifdef RC_BRINGUP
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {   // ~2 s at 2 GHz
      printf("rangeclip_b200: mbarrier timeout tag=%d block=%d thread=%d parity=%u\n", tag, (int)blockIdx.x,
             (int)threadIdx.x, parity);
      __trap();
    }
  }
#else
  (void)tag;
  while (!mbar_try_wait(bar, parity)) {}
#endif
}

// ---- proxies / fences -------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---- TMA --------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// ---- L2 eviction-priority hints ---------------------------------------------------------------
__device__ __forceinline__ void tma_load_3d_hint(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, uint64_t pol);
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void tma_load_3d_hint(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "l"(pol)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_2sm_hint(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                                     uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1), "r"(c2), "l"(pol)
      : "memory");
}
__device__ __forceinline__ void tma_store_3d_hint(const CUtensorMap* m, const void* src, int c0, int c1, int c2, uint64_t pol) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3, %4}], [%1], %5;" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "l"(pol)
               : "memory");
}
// bulk tensor store that ADDS the shared-memory box to global memory (element type from the tensor map: bf16 here); the
// read-modify-write happens in the L2
__device__ __forceinline__ void tma_reduce_add_3d(const CUtensorMap* m, const void* src, int c0, int c1, int c2) {
  asm volatile("cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
// L2 prefetch of one box (no shared-memory destination, no completion tracking)
__device__ __forceinline__ void tma_prefetch_3d(const CUtensorMap* m, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(reinterpret_cast<uint64_t>(m)), "r"(c0),
               "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// all but the most recently committed bulk group have finished READING their shared-memory source
__device__ __forceinline__ void tma_store_wait_read0_keep1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }

// ---- TMEM -------------------------------------------------------------------------------------
template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem) {   // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {      // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp receives lane (taddr.lane + i)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// 16 lanes x 32 consecutive 32-bit columns in the accumulator-fragment layout of mma.m16n8: for column group g (8 columns),
// r[4g+0], r[4g+1] = (lane taddr.lane + t/4, columns 8g + 2(t%4), +1) and r[4g+2], r[4g+3] = the same columns of lane + 8
__device__ __forceinline__ void tmem_ld_16x256b_x4(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// four 8x8 b16 matrices, transposed on the way: thread t supplies the address of row (t & 7) of matrix (t >> 3) and
// receives / provides, per matrix, the pair (column t/4 of rows 2(t%4), 2(t%4)+1)
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t saddr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(saddr)
               : "memory");
}
__device__ __forceinline__ void stmatrix_x4_trans(uint32_t saddr, const uint32_t (&r)[4]) {
  asm volatile("stmatrix.sync.aligned.m8n8.x4.trans.shared.b16 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(r[0]), "r"(r[1]),
               "r"(r[2]), "r"(r[3])
               : "memory");
}
// 32 lanes x 16 columns register -> TMEM store (thread i writes lane taddr.lane + i) and its completion wait
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// wait that also "redefines" the destination registers of an earlier, still outstanding tcgen05.ld, so that the
// compiler cannot schedule a use of them ahead of the wait (for loads issued early to overlap with other work)
__device__ __forceinline__ void tmem_ld_wait32(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]),
                 "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]),
                 "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}

// ---- descriptors ------------------------------------------------------------------------------
// Shared-memory matrix descriptor (64-bit): start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) |
// version=1 [46,48) | base_offset [49,52) | layout_type [61,64) (2 = SWIZZLE_128B).
__host__ __device__ constexpr uint64_t make_smem_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46) | (2ull << 61);
}
// K-major operand tile stored as rows of 64 bf16 (128 B) with the 128-byte swizzle: 8-row groups
// are 1024 B apart (SBO); LBO is unused for swizzled K-major layouts.
__device__ __forceinline__ uint64_t desc_kmajor_sw128(uint32_t smem_addr) {
  return make_smem_desc_sw128(smem_addr, 16, 1024);
}
// MN-major operand tile: rows are K indices, each row holds 64 consecutive MN elements (128 B);
// 8 K-rows form one swizzle atom (1024 B, SBO between atoms along K); LBO = byte distance between
// consecutive 64-element groups along MN.
__device__ __forceinline__ uint64_t desc_mnmajor_sw128(uint32_t smem_addr, uint32_t mn_group_stride_bytes) {
  return make_smem_desc_sw128(smem_addr, mn_group_stride_bytes, 1024);
}
// Instruction descriptor, kind::f16, bf16 x bf16 -> f32:
// c_format[4,6)=1(F32) a_format[7,10)=1(BF16) b_format[10,13)=1(BF16) a_major[15] b_major[16]
// n_dim[17,23)=N>>3 m_dim[24,29)=M>>4
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread.
__device__ __forceinline__ void mma_bf16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives when all previously issued tcgen05 async ops of this thread have completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}


// ---- thread-block clusters / CTA pairs (cta_group::2) --------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.aligned;" ::: "memory");
}
// shared::cluster address of `p` (a shared::cta pointer of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(const void* p, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
  return r;
}
// Remote arrive with the default (release, CTA scope) semantics: a plain SYNCS.ARRIVE over the cluster network.
// (`.release.cluster` compiles to MEMBAR.ALL.GPU, which drains every global load / store the thread has in
// flight -- fatal for roles that stream global memory.)  Data published with it must be in the ARRIVING CTA's
// shared memory (+ fence.proxy.async when the tensor cores read it); data for the peer CTA goes through
// st_async_remote_v2 below, which carries its own completion.
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// 8-byte store into the peer CTA's shared memory; completes 8 transaction bytes on the peer's mbarrier
__device__ __forceinline__ void st_async_remote_v2(uint32_t cluster_addr, uint32_t a, uint32_t b, uint32_t cluster_mbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.b32 [%0], {%1, %2}, [%3];" ::"r"(cluster_addr),
               "r"(a), "r"(b), "r"(cluster_mbar)
               : "memory");
}
// 4-byte variant
__device__ __forceinline__ void st_async_remote_b32(uint32_t cluster_addr, uint32_t a, uint32_t cluster_mbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(cluster_addr), "r"(a),
               "r"(cluster_mbar)
               : "memory");
}
// packed bf16x2 arithmetic on raw 32-bit registers
__device__ __forceinline__ uint32_t bf2_mul(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("mul.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
__device__ __forceinline__ uint32_t bf2_fma(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("fma.rn.bf16x2 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
// wait with cluster-scope acquire (barriers that receive remote arrivals / guard remotely written data)
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(kSuspendHintNs)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity, int tag) {
#ifdef RC_BRINGUP
  if (mbar_try_wait_cluster(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait_cluster(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {
      printf("rangeclip_b200: cluster mbarrier timeout tag=%d block=%d thread=%d parity=%u\n", tag, (int)blockIdx.x,
             (int)threadIdx.x, parity);
      __trap();
    }
  }
#else
  (void)tag;
  while (!mbar_try_wait_cluster(bar, parity)) {}
#endif
}
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;   // shared::cluster address of the same offset in CTA 0 of the pair
// 2-SM TMA loads: issued by either CTA of the pair into ITS OWN shared memory; the transaction bytes are
// credited to the mbarrier at the same offset in the LEADER CTA (rank 0).
__device__ __forceinline__ void tma_load_2d_2sm(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_2sm(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* dst_smem) {   // one warp in EACH CTA of the pair
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
// D[tmem, both CTAs] (+)= A[smem, M = 256: 128 rows per CTA] * B[smem, N split: N/2 rows per CTA]; leader thread only
__device__ __forceinline__ void mma_bf16_ss_2sm(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// TS mode: D[tmem, both CTAs] (+)= A[TMEM of each CTA: its 128 rows, packed bf16 pairs, 8 columns per 16 k] *
// B[smem, N split: N/2 rows per CTA].  A must be K-major (operands in tensor memory cannot be transposed).
__device__ __forceinline__ void mma_bf16_ts_2sm(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                                uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (once all prior MMAs of this thread completed) on the mbarrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void mma_commit_2sm(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"((uint16_t)3)
      : "memory");
}

}  // namespace umma

// ---- host (umma.cu): tensor-map encoding through the driver entry point (no -lcuda link dependency) ------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiled get_encode_tiled();

// bf16 tensor map, 128-byte swizzle, zero OOB fill.  dims/strides innermost first; strides[0] is
// implied (2 bytes); `rank` in {2,3}.
int make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box, const char* what);

}  // namespace rc
