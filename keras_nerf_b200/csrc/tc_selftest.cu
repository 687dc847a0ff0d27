// Single-tile tcgen05 self-test: D[128 x N] = A[128 x K] * B[N x K]^T with operands in the chunk-major
// layout of tc_ptx.cuh, either K-major (forward / dgrad form) or MN-major (weight-gradient form, reduction
// dimension = rows of the stored blobs).  Used by tests/test_gpu_tc.py to pin the UMMA descriptor encoding
// independently of the fused MLP kernels.
#include "common.cuh"
#include "tc_ptx.cuh"

namespace knerf {
using namespace tc;

// mode 0: A blob [K/8][128][8], B blob [K/8][N][8]           (K-major, K = reduction)
// mode 1: A blob [128/8][K][8], B blob [N/8][K][8]           (MN-major, K = rows of the blobs)
// mode 2: A blob [128/16][K][16] e4m3, B blob [N/16][K][16] e5m2   (MN-major fp8, kind::f8f6f4: the weight-gradient
//         GEMM over fp8 records)
__global__ void __launch_bounds__(128) umma_selftest_kernel(int mode, const uint8_t* __restrict__ a_blob,
                                                            const uint8_t* __restrict__ b_blob, int N, int K,
                                                            float* __restrict__ d_out) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_load, bar_mma;
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t esz = mode == 2 ? 1u : 2u;
  const uint32_t a_bytes = 128u * K * esz, b_bytes = (uint32_t)N * K * esz;
  uint8_t* sa = smem;
  uint8_t* sb = smem + a_bytes;
  if (tid == 0) {
    mbar_init(&bar_load, 1);
    mbar_init(&bar_mma, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc<256>(&tmem_base_s);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  if (tid == 0) {
    mbar_arrive_expect_tx(&bar_load, a_bytes + b_bytes);
    tma_load_1d(sa, a_blob, a_bytes, &bar_load);
    tma_load_1d(sb, b_blob, b_bytes, &bar_load);
    mbar_wait(&bar_load, 0);
    tc_fence_after();
    if (mode == 2) {
      const uint32_t idesc8 = umma_idesc_f8(128, N, kE4M3, kE5M2, 1, 1);
      for (int k = 0; k < K / 32; ++k) {   // 32 k per instruction = 32 rows x 16 B of every chunk
        const uint64_t da = umma_smem_desc(smem_u32(sa) + k * 512, 128, K * 16);
        const uint64_t db = umma_smem_desc(smem_u32(sb) + k * 512, 128, K * 16);
        umma_f8(tmem, da, db, idesc8, k > 0 ? 1u : 0u);
      }
    }
    const uint32_t idesc = umma_idesc_bf16(128, N, mode, mode);
    for (int k = 0; k < (mode == 2 ? 0 : K / 16); ++k) {
      uint64_t da, db;
      if (mode == 0) {
        da = umma_smem_desc(smem_u32(sa) + k * 2 * (128 * 16), 128 * 16, 128);
        db = umma_smem_desc(smem_u32(sb) + k * 2 * (N * 16), N * 16, 128);
      } else {
        da = umma_smem_desc(smem_u32(sa) + k * 256, 128, K * 16);
        db = umma_smem_desc(smem_u32(sb) + k * 256, 128, K * 16);
      }
      umma_bf16(tmem, da, db, idesc, k > 0 ? 1u : 0u);
    }
    umma_commit(&bar_mma);
  }
  mbar_wait(&bar_mma, 0);
  tc_fence_after();
  const int row = warp * 32 + lane;
  for (int c0 = 0; c0 < N; c0 += 32) {
    float v[32];
    tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + c0, v);
#pragma unroll
    for (int i = 0; i < 32; ++i)
      if (c0 + i < N) d_out[(size_t)row * N + c0 + i] = v[i];
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc<256>(tmem);
}

// 2-CTA form: D[256 x N] = A[256 x K] * B[N x K]^T with one tcgen05.mma.cta_group::2 per K=16 step.
// CTA c of the pair holds A rows [128c, 128c+128) and B rows [c*N/2, (c+1)*N/2) (K-major, chunk-major blobs
// a_blob = [2][K/8][128][8], b_blob = [2][K/8][N/2][8]); each CTA reads its own 128 accumulator lanes.
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128)
umma_selftest2_kernel(const uint8_t* __restrict__ a_blob, const uint8_t* __restrict__ b_blob, int N, int K,
                      float* __restrict__ d_out) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_load, bar_mma;
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t cta = cluster_ctarank();
  const uint32_t a_bytes = 128u * K * 2u, b_bytes = (uint32_t)(N / 2) * K * 2u;
  uint8_t* sa = smem;
  uint8_t* sb = smem + a_bytes;
  if (tid == 0) {
    mbar_init(&bar_load, 1);
    mbar_init(&bar_mma, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc_2cta<256>(&tmem_base_s);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  if (tid == 0) {
    mbar_arrive_expect_tx(&bar_load, a_bytes + b_bytes);
    tma_load_1d(sa, a_blob + (size_t)cta * a_bytes, a_bytes, &bar_load);
    tma_load_1d(sb, b_blob + (size_t)cta * b_bytes, b_bytes, &bar_load);
    mbar_wait(&bar_load, 0);
  }
  cluster_sync_all();   // both CTAs' operands have landed
  if (cta == 0 && tid == 0) {
    tc_fence_after();
    const uint32_t idesc = umma_idesc_bf16(256, N, 0, 0);
    for (int k = 0; k < K / 16; ++k) {
      const uint64_t da = umma_smem_desc(smem_u32(sa) + k * 2 * (128 * 16), 128 * 16, 128);
      const uint64_t db = umma_smem_desc(smem_u32(sb) + k * 2 * ((N / 2) * 16), (N / 2) * 16, 128);
      umma_bf16_2cta(tmem, da, db, idesc, k > 0 ? 1u : 0u);
    }
    umma_commit_2cta(&bar_mma, 3);
  }
  mbar_wait_cluster(&bar_mma, 0);
  tc_fence_after();
  const int row = (int)cta * 128 + warp * 32 + lane;
  for (int c0 = 0; c0 < N; c0 += 32) {
    float v[32];
    tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + c0, v);
#pragma unroll
    for (int i = 0; i < 32; ++i)
      if (c0 + i < N) d_out[(size_t)row * N + c0 + i] = v[i];   // (N = 16: the load also returns 16 unused columns)
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 0) tmem_dealloc_2cta<256>(tmem);
}

}  // namespace knerf

using namespace knerf;

extern "C" int knerf_selftest_umma2(const void* a_blob, const void* b_blob, int N, int K, float* d_out, void* stream) {
  KN_CHECK_ARG(a_blob && b_blob && d_out, "knerf_selftest_umma2: null pointer");
  KN_CHECK_ARG(N % 16 == 0 && N >= 16 && N <= 256 && K % 16 == 0 && K >= 16 && K <= 256,
               "knerf_selftest_umma2: N in 16..256 step 16, K in 16..256 step 16");
  const size_t smem = (size_t)(128 + N / 2) * K * 2;
  KN_CUDA(cudaFuncSetAttribute(umma_selftest2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  umma_selftest2_kernel<<<2, 128, smem, (cudaStream_t)stream>>>((const uint8_t*)a_blob, (const uint8_t*)b_blob, N, K,
                                                                d_out);
  KN_LAUNCH_CHECK();
  return KNERF_OK;
}

extern "C" int knerf_selftest_umma(int mode, const void* a_blob, const void* b_blob, int N, int K, float* d_out,
                                   void* stream) {
  KN_CHECK_ARG(a_blob && b_blob && d_out, "knerf_selftest_umma: null pointer");
  if (mode == 2) {
    KN_CHECK_ARG(N % 16 == 0 && N >= 16 && N <= 256 && K % 32 == 0 && K >= 32 && K <= 256,
                 "knerf_selftest_umma: mode 2, N in 16..256 step 16, K in 32..256 step 32");
  } else {
    KN_CHECK_ARG((mode == 0 || mode == 1) && N % 32 == 0 && N >= 32 && N <= 256 && K % 16 == 0 && K >= 16 && K <= 256,
                 "knerf_selftest_umma: mode 0/1, N in 32..256 step 32, K in 16..256 step 16");
  }
  const size_t smem = (size_t)(128 + N) * K * (mode == 2 ? 1 : 2);
  KN_CUDA(cudaFuncSetAttribute(umma_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  umma_selftest_kernel<<<1, 128, smem, (cudaStream_t)stream>>>(mode, (const uint8_t*)a_blob, (const uint8_t*)b_blob, N,
                                                               K, d_out);
  KN_LAUNCH_CHECK();
  return KNERF_OK;
}
