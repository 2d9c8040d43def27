// Bring-up GEMMs: one tile of C = A B^T through the same TMA / descriptor / tcgen05 / TMEM building blocks as the fused
// kernels, checked against torch.matmul by tests/test_gpu_parity.py.  Compiled only into the bring-up library
// (librangeclip_b200_bringup.so, -DRC_BRINGUP); the shipped library holds none of these kernels.
//   debug_umma_gemm_kernel         C[128][N], one CTA; descriptor variants for the K-major / MN-major A operand
//   debug_umma_gemm_2sm_kernel     C[256][N], a CTA pair (cta_group::2): A rows split 128/128, B rows N/2 / N/2
//   debug_umma_gemm_ts_2sm_kernel  the CTA-pair GEMM with A as a tensor-memory operand (TS mode), written by the threads
//                                  with tcgen05.st (packed bf16 pairs)
#include "common.cuh"
#include "umma.cuh"

namespace rc {

using namespace umma;

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

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128, 1)
debug_umma_gemm_ts_2sm_kernel(const __grid_constant__ CUtensorMap map_b, const __nv_bfloat16* __restrict__ a, int N, int Kd,
                              float* __restrict__ c) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sbm = smem;              // Kd/64 chunks of own N/2 rows of B (<= 4 x 16 KB)
  DebugBars* bars = reinterpret_cast<DebugBars*>(smem + 65536);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int nh = N / 2;
  if (threadIdx.x == 0) {
    mbar_init(&bars->full, 1);
    mbar_init(&bars->done, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_2sm<512>(&bars->tmem_base);
  tc_fence_before();
  cluster_sync();
  tc_fence_after();
  const uint32_t tmem = bars->tmem_base;
  const int row = warp * 32 + lane;
  {
    // own row of A as packed pairs: column 256 + j holds k = 2j (low half), 2j + 1 (high half)
    const uint32_t* src = reinterpret_cast<const uint32_t*>(a + ((int64_t)rank * 128 + row) * Kd);
    for (int cc = 0; cc < Kd / 32; ++cc) {
      uint32_t v[16];
      for (int i = 0; i < 16; ++i) v[i] = src[cc * 16 + i];
      tmem_st_32x16(tmem + ((uint32_t)(warp * 32) << 16) + 256 + cc * 16, v);
    }
    tmem_st_wait();
  }
  tc_fence_before();
  cluster_sync();
  tc_fence_after();
  if (threadIdx.x == 0) {
    const int nck = Kd / 64;
    if (rank == 0) mbar_arrive_expect_tx(&bars->full, 2 * nck * nh * 128);
    for (int ck = 0; ck < nck; ++ck) tma_load_2d_2sm(sbm + ck * nh * 128, &map_b, &bars->full, ck * 64, (int)rank * nh);
    if (rank == 0) {
      const uint32_t idesc = make_idesc_bf16(256, N, 0, 0);
      mbar_wait(&bars->full, 0, 210);
      tc_fence_after();
      for (int ck = 0; ck < nck; ++ck)
        for (int ks = 0; ks < 4; ++ks)
          mma_bf16_ts_2sm(tmem, tmem + 256 + (ck * 4 + ks) * 8, desc_kmajor_sw128(smem_u32(sbm) + ck * nh * 128 + ks * 32), idesc,
                          (ck | ks) != 0);
      mma_commit_2sm(&bars->done);
    }
    mbar_wait(&bars->done, 0, 211);
  }
  __syncthreads();
  tc_fence_after();
  for (int cc = 0; cc < N / 32; ++cc) {
    uint32_t r[32];
    tmem_ld_32x32(tmem + ((uint32_t)(warp * 32) << 16) + cc * 32, r);
    tmem_ld_wait();
    for (int i = 0; i < 32; ++i) c[((int64_t)rank * 128 + row) * N + cc * 32 + i] = __uint_as_float(r[i]);
  }
  tc_fence_before();
  cluster_sync();
  if (warp == 1) { tc_fence_after(); tmem_dealloc_2sm<512>(tmem); }
}

}  // namespace rc

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

extern "C" int rc_debug_umma_gemm_ts_2sm(const void* a_bf16, const void* b_bf16, int N, int Kd, float* c, void* stream) {
  RC_REQUIRE(a_bf16 && b_bf16 && c, "rc_debug_umma_gemm_ts_2sm: null pointer");
  RC_REQUIRE(N >= 64 && N <= 256 && N % 64 == 0 && Kd >= 64 && Kd <= 256 && Kd % 64 == 0, "rc_debug_umma_gemm_ts_2sm: bad shape N=%d Kd=%d", N, Kd);
  CUtensorMap mb;
  int rcode;
  {
    const uint64_t bdims[2] = {(uint64_t)Kd, (uint64_t)N}, str[2] = {2, (uint64_t)Kd * 2};
    const uint32_t bbox[2] = {64, (uint32_t)(N / 2)};
    if ((rcode = rc::make_tmap_bf16(&mb, b_bf16, 2, bdims, str, bbox, "debug ts B"))) return rcode;
  }
  const int smem = 65536 + 64;
  cudaError_t e = cudaFuncSetAttribute(rc::debug_umma_gemm_ts_2sm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return rc::fail(RC_ERR_CUDA, "rc_debug_umma_gemm_ts_2sm: smem opt-in: %s", cudaGetErrorString(e));
  rc::debug_umma_gemm_ts_2sm_kernel<<<2, 128, smem, (cudaStream_t)stream>>>(mb, (const __nv_bfloat16*)a_bf16, N, Kd, c);
  return rc::check_launch("rc_debug_umma_gemm_ts_2sm");
}
