// Microbenchmark: raw issue/execute rate of tcgen05.mma from shared-memory operands in the library's chunk-major
// (SWIZZLE_NONE) layout, 1-CTA (M=128) and cta_group::2 (M=256), with and without a tcgen05.commit per K=32 stage.
// rate_f8_kernel: kind::f8f6f4 (e4m3 x e5m2) at the weight-gradient kernel's shapes -- M 128, K 32, N 256 / 128, both
// operands MN-major with LBO 128 B / SBO 2 KB exactly as tc_wgrad_kernel builds them (or the same bytes K-major), issued
// by one thread or by two threads into disjoint accumulators.
// build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -I keras_nerf_b200/csrc -o benchmarks/micro/umma_rate benchmarks/micro/umma_rate.cu
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>
#include "tc_ptx.cuh"
using namespace knerf::tc;

constexpr int kA = 128 * 256 * 2;      // one A tile [128 x 256] bf16
constexpr int kStage = 256 * 32 * 2;   // one full-N weight stage (K = 32)

template <bool TWO, bool MN = false>
__global__ void __launch_bounds__(128) rate_kernel(int n_stages, int N, int commit_every, long long* out) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_done, bar_full, bar_stage[8];
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t cta = TWO ? cluster_ctarank() : 0u;
  for (int i = tid; i < (kA + 4 * kStage) / 4; i += 128) reinterpret_cast<uint32_t*>(smem)[i] = 0x3c003c00u + i;
  if (tid == 0) {
    mbar_init(&bar_done, 1);
    mbar_init(&bar_full, 1);
    for (int i = 0; i < 8; ++i) mbar_init(&bar_stage[i], 1);
    fence_mbar_init();
  }
  if (warp == 0) { if (TWO) tmem_alloc_2cta<512>(&tmem_base_s); else tmem_alloc<512>(&tmem_base_s); }
  fence_async_smem();
  tc_fence_before();
  if (TWO) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  long long t0 = 0, t1 = 0, t2 = 0;
  if (cta == 0 && tid == 0) {
    const uint32_t idesc = umma_idesc_bf16(TWO ? 256 : 128, N, MN ? 1 : 0, MN ? 1 : 0);
    const uint32_t chunk_b = (uint32_t)(TWO ? N / 2 : N) * 16;
    t0 = clock64();
    for (int s = 0; s < n_stages; ++s) {
      const uint32_t a_base = smem_u32(smem) + (MN ? 0 : (s % 8) * 4 * 2048);
      const uint32_t b_base = smem_u32(smem) + (MN ? 32768 : kA + (s % 4) * kStage);
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        // MN: the weight-gradient form (tc_ptx.cuh): K = rows of the blobs, LBO = 128 B (next 8 k), SBO = 2 KB (next 8 m|n)
        const uint64_t da = MN ? umma_smem_desc(a_base + j * 256, 128, 2048) : umma_smem_desc(a_base + j * 2 * 2048, 2048, 128);
        const uint64_t db = MN ? umma_smem_desc(b_base + j * 256, 128, 2048) : umma_smem_desc(b_base + j * 2 * chunk_b, chunk_b, 128);
        if (TWO) umma_bf16_2cta(tmem + (s & 256), da, db, idesc, s > 0);
        else umma_bf16(tmem + (s & 256), da, db, idesc, s > 0);
      }
      // commit_every is a bit mask here: 1 = commit per stage, 2 = wait on an (already complete) barrier per stage,
      // 4 = tcgen05.fence::after_thread_sync per stage, 8 = commit every 2nd stage only
      if (commit_every & 2) mbar_wait(&bar_full, 1);
      if (commit_every & 4) tc_fence_after();
      if ((commit_every & 1) || ((commit_every & 8) && (s & 1))) {
        if (TWO) umma_commit_2cta(&bar_stage[s % 8], 3); else umma_commit(&bar_stage[s % 8]);
      }
    }
    t1 = clock64();
    if (TWO) umma_commit_2cta(&bar_done, 3); else umma_commit(&bar_done);
  }
  if (TWO) mbar_wait_cluster(&bar_done, 0); else mbar_wait(&bar_done, 0);
  t2 = clock64();
  tc_fence_after();
  if (cta == 0 && tid == 0) { out[blockIdx.x * 2] = t1 - t0; out[blockIdx.x * 2 + 1] = t2 - t0; }
  tc_fence_before();
  if (TWO) cluster_sync_all(); else __syncthreads();
  if (warp == 0) { if (TWO) tmem_dealloc_2cta<512>(tmem); else tmem_dealloc<512>(tmem); }
}

template <bool TWO, bool MN = false>
void run(int grid, int n_stages, int N, int commit_every) {
  long long* d;
  cudaMalloc(&d, 148 * 2 * sizeof(long long));
  cudaMemset(d, 0, 148 * 2 * sizeof(long long));
  const size_t smem = kA + 4 * kStage;
  cudaFuncSetAttribute(rate_kernel<TWO, MN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaLaunchConfig_t cfg{};
  cudaLaunchAttribute attr[1];
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(128); cfg.dynamicSmemBytes = smem;
  if (TWO) {
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
  }
  for (int rep = 0; rep < 2; ++rep) {
    cudaError_t e = cudaLaunchKernelEx(&cfg, rate_kernel<TWO, MN>, n_stages, N, commit_every, d);
    if (e != cudaSuccess || (e = cudaDeviceSynchronize()) != cudaSuccess) { printf("error: %s\n", cudaGetErrorString(e)); exit(1); }
  }
  long long h[296];
  cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost);
  double issue = 0, total = 0; int n = 0;
  for (int b = 0; b < grid; b += (TWO ? 2 : 1)) { issue += h[b * 2]; total += h[b * 2 + 1]; ++n; }
  printf("%s grid %3d N %3d stages %5d mode %2d: issue %.1f cyc/MMA, complete %.1f cyc/MMA (floor %d)\n",
         MN ? "1-CTA M=128 MN-major A and B" : TWO ? "2-CTA M=256" : "1-CTA M=128", grid, N, n_stages, commit_every, issue / n / (2.0 * n_stages),
         total / n / (2.0 * n_stages), N / 2);
  cudaFree(d);
}

// fp8: A = [8 chunks][128 k][16] (16 KB), B = [N/16 chunks][128 k][16] (N = 256: 32 KB) -- one weight-gradient tile of
// 128 samples, 4 MMAs of K = 32.  K-major: the same 48 KB as [8 k-chunks][rows][16].  LAYOUT: 0 both MN-major, 1 both
// K-major, 2 A MN-major / B K-major, 3 A K-major / B MN-major.  mode bit 0: tcgen05.commit per
// 4 MMAs; bit 1: mbarrier.try_wait (on an already completed phase) per 4 MMAs -- the issuer loop of tc_wgrad_kernel.
template <int LAYOUT>
__global__ void __launch_bounds__(64) rate_f8_kernel(int n_mma, int N, int issuers, int mode, long long* out) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_done[2], bar_full, bar_stage[2];
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5;
  for (int i = tid; i < 49152 / 4; i += 64) reinterpret_cast<uint32_t*>(smem)[i] = 0x38383838u ^ (i & 0x07070707u);
  if (tid == 0) {
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_done[i], 1); mbar_init(&bar_stage[i], 1); }
    mbar_init(&bar_full, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc<512>(&tmem_base_s);
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const int me = warp;
  if ((tid & 31) == 0 && me < issuers) {
    constexpr bool KA = LAYOUT == 1 || LAYOUT == 3, KB = LAYOUT == 1 || LAYOUT == 2;
    const uint32_t idesc = umma_idesc_f8(128, N, kE4M3, kE5M2, KA ? 0 : 1, KB ? 0 : 1);
    const uint32_t a_base = smem_u32(smem), b_base = smem_u32(smem) + 16384;
    const long long t0 = clock64();
    for (int s = 0; s < n_mma; s += 4) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint64_t da = KA ? umma_smem_desc(a_base + k * 2 * 2048, 2048, 128) : umma_smem_desc(a_base + k * 512, 128, 2048);
        const uint64_t db = KB ? umma_smem_desc(b_base + k * 2 * N * 16, N * 16, 128) : umma_smem_desc(b_base + k * 512, 128, 2048);
        umma_f8(tmem + me * 256, da, db, idesc, (s > 0 || k > 0) ? 1u : 0u);
      }
      if (mode & 2) mbar_wait(&bar_full, 1);
      if (mode & 1) umma_commit(&bar_stage[me]);
    }
    const long long t1 = clock64();
    umma_commit(&bar_done[me]);
    mbar_wait(&bar_done[me], 0);
    const long long t2 = clock64();
    out[(blockIdx.x * 2 + me) * 2] = t1 - t0;
    out[(blockIdx.x * 2 + me) * 2 + 1] = t2 - t0;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc<512>(tmem);
}

template <int LAYOUT>
void run_f8(int n_mma, int N, int issuers, int mode) {
  constexpr int grid = 148;
  long long* d;
  cudaMalloc(&d, grid * 4 * sizeof(long long));
  cudaMemset(d, 0, grid * 4 * sizeof(long long));
  cudaFuncSetAttribute(rate_f8_kernel<LAYOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 49152);
  for (int rep = 0; rep < 2; ++rep) {
    rate_f8_kernel<LAYOUT><<<grid, 64, 49152>>>(n_mma, N, issuers, mode, d);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess || (e = cudaDeviceSynchronize()) != cudaSuccess) { printf("error: %s\n", cudaGetErrorString(e)); exit(1); }
  }
  long long h[grid * 4];
  cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost);
  double issue = 0, total = 0;
  for (int b = 0; b < grid; ++b) {
    double t = 0;
    for (int x = 0; x < issuers; ++x) { issue += h[(b * 2 + x) * 2]; t = h[(b * 2 + x) * 2 + 1] > t ? h[(b * 2 + x) * 2 + 1] : t; }
    total += t;
  }
  // issue: cycles one issuer spends per MMA it issues; complete: SM time per MMA, all issuers' MMAs counted
  printf("f8 e4m3 x e5m2 %s M=128 N %3d K 32, %d issuer(s), commit %d wait %d: issue %.1f cyc/MMA, complete %.1f cyc/MMA"
         " (floor %d)\n", LAYOUT == 0 ? "A, B MN-major" : LAYOUT == 1 ? "A, B K-major " : LAYOUT == 2 ? "A MN, B K    " : "A K, B MN    ", N, issuers, mode & 1, (mode >> 1) & 1,
         issue / grid / issuers / n_mma, total / grid / ((double)issuers * n_mma), N / 2);
  cudaFree(d);
}

int main() {
  for (int mode : {0, 1, 2, 4, 3, 7, 8, 14}) {
    run<false>(148, 4096, 256, mode);
    run<true>(148, 4096, 256, mode);
  }
  run<true>(148, 4096, 128, 7);
  // weight-gradient form: both operands MN-major, N = 128 (floor 64) and N = 256
  run<false>(148, 4096, 128, 0);
  run<false, true>(148, 4096, 128, 0);
  run<false, true>(148, 4096, 256, 0);
  // kind::f8f6f4 at the shapes of tc_wgrad_kernel (fp8 records)
  for (int N : {256, 128})
    for (int issuers : {1, 2})
      for (int mode : {0, 3}) {
        run_f8<0>(8192, N, issuers, mode);
        run_f8<1>(8192, N, issuers, mode);
      }
  run_f8<2>(8192, 256, 1, 0);
  run_f8<3>(8192, 256, 1, 0);
  return 0;
}
