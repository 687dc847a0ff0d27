// a6 (KNERF_FP32_TC mode): the fp32 NeRF MLP on Blackwell tensor cores (keras_nerf/model/nerf/mlp.py:29-50; the
// reference is fp32 end to end: mlp.py:11-27 sets no mixed-precision policy).
//
// tcgen05 has no fp32 x fp32 MMA.  Every fp32 operand x is therefore split into THREE bf16 values
//     x = x1 + x2 + x3,   x1 = bf16(x), x2 = bf16(x - x1), x3 = bf16(x - x1 - x2)      (24 mantissa bits in total)
// and a product a*b is formed as the six leading terms  a1 b1 + a1 b2 + a2 b1 + a1 b3 + a2 b2 + a3 b1
// (the dropped ones are below 2^-24 |a b|), each an exact bf16 x bf16 product accumulated in fp32 in TMEM: fp32-grade
// results at one sixth of the bf16 tensor rate -- ~9x what the SIMT FFMA path reaches (mlp_fp32.cu).
//
// Two kernels, both one GEMM per Dense layer with fp32 activations in HBM (like the SIMT mode, whose host code
// -- fp32_forward_core / fp32_backward_core -- drives them):
//   tcx_gemm_kernel   C[M,N] = epi(A1 B1 + A2 B2 + bias): forward layers and dgrad.  A tile: fp32 rows loaded and
//                     split by the compute warps into the chunk-major K-major layout of tc_ptx.cuh; B: the weights,
//                     split ONCE per call into operand blobs (tcx_pack_kernel) and streamed by bulk copies.
//   tcx_wgrad_kernel  dW[K,N] += A[M,K]^T Z[M,N], reduction over samples: both operands split on the fly into the
//                     MN-major form (same bytes, other axis), accumulators resident in TMEM over a slab of samples.
#include "mlp_fp32.cuh"
#include "tc_ptx.cuh"

namespace knerf {
using namespace tc;

namespace {

constexpr int kXThreads = 320;          // weight-gradient kernel: warps 0-7 compute (split + flush), warps 8 and 9 = MMA
                                        // issue (feature rows 0..127 / 128..255: one issuer per accumulator)
// the six products, ordered from the smallest terms to the largest (the order only matters for rounding)
__device__ __constant__ int8_t kProdA[6] = {2, 1, 0, 1, 0, 0};
__device__ __constant__ int8_t kProdB[6] = {0, 1, 2, 0, 1, 0};

// 8 consecutive fp32 -> three 16-byte vectors of bf16 (x1 | x2 | x3), element e in half (e & 1) of word e >> 1
__device__ __forceinline__ void split3x8(const float (&x)[8], uint4& p1, uint4& p2, uint4& p3) {
  uint32_t w1[4], w2[4], w3[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float a = x[2 * i], b = x[2 * i + 1];
    w1[i] = pack_bf16x2(a, b);
    const float ra = a - bf16_lo(w1[i]), rb = b - bf16_hi(w1[i]);      // exact
    w2[i] = pack_bf16x2(ra, rb);
    w3[i] = pack_bf16x2(ra - bf16_lo(w2[i]), rb - bf16_hi(w2[i]));
  }
  p1 = make_uint4(w1[0], w1[1], w1[2], w1[3]);
  p2 = make_uint4(w2[0], w2[1], w2[2], w2[3]);
  p3 = make_uint4(w3[0], w3[1], w3[2], w3[3]);
}

// 4 consecutive fp32 -> three 8-byte vectors of bf16 (x1 | x2 | x3)
__device__ __forceinline__ void split3x4(const float4 x, uint2& p1, uint2& p2, uint2& p3) {
  const uint32_t a1 = pack_bf16x2(x.x, x.y), b1 = pack_bf16x2(x.z, x.w);
  const float r0 = x.x - bf16_lo(a1), r1 = x.y - bf16_hi(a1), r2 = x.z - bf16_lo(b1), r3 = x.w - bf16_hi(b1);   // exact
  const uint32_t a2 = pack_bf16x2(r0, r1), b2 = pack_bf16x2(r2, r3);
  p1 = make_uint2(a1, b1);
  p2 = make_uint2(a2, b2);
  p3 = make_uint2(pack_bf16x2(r0 - bf16_lo(a2), r1 - bf16_hi(a2)), pack_bf16x2(r2 - bf16_lo(b2), r3 - bf16_hi(b2)));
}

// 4 fp32 of row `grow`, reduction columns k0 .. k0 + 3 of source A (zero beyond M / K)
__device__ __forceinline__ float4 load_a4(const float* __restrict__ A, int lda, int K, int64_t grow, int64_t M, int k0) {
  if (grow < M && k0 + 4 <= K && (lda & 3) == 0 && (reinterpret_cast<uintptr_t>(A) & 15) == 0)
    return __ldg(reinterpret_cast<const float4*>(A + grow * lda + k0));
  float x[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) x[e] = (grow < M && k0 + e < K) ? __ldg(A + grow * lda + k0 + e) : 0.f;
  return make_float4(x[0], x[1], x[2], x[3]);
}

// ---- weight operand blobs -------------------------------------------------------------------------------------
// B[n][k] (n < N outputs, k < K reduction) = src[k * ld + n] (TRANS = false: a Keras kernel [in,out] used forward) or
// src[n * ld + k] (TRANS = true: the same kernel used by dgrad).  Blob: [K16 steps][3 splits][2 chunks][N][8] bf16, zero
// beyond K, so that one step's stage is ONE contiguous bulk copy.  One thread per 16-byte vector (all three splits).

__global__ void __launch_bounds__(256) tcx_pack_kernel(const float* __restrict__ src, int ld, int N, int K, int trans,
                                                       uint8_t* __restrict__ blob) {
  const int ksteps = (K + 15) / 16;
  const int total = ksteps * 2 * N;
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < total; v += gridDim.x * blockDim.x) {
    const int n = v % N, c = (v / N) & 1, ks = v / (2 * N);
    float x[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int k = ks * 16 + c * 8 + e;
      x[e] = (k < K) ? (trans ? src[(int64_t)n * ld + k] : src[(int64_t)k * ld + n]) : 0.f;
    }
    uint4 p1, p2, p3;
    split3x8(x, p1, p2, p3);
    uint8_t* base = blob + (size_t)ks * 96 * N + (size_t)(c * N + n) * 16;
    *reinterpret_cast<uint4*>(base) = p1;
    *reinterpret_cast<uint4*>(base + 32 * N) = p2;
    *reinterpret_cast<uint4*>(base + 64 * N) = p3;
  }
}

// ---- C = epi(A1 B1 + A2 B2 + bias) ----------------------------------------------------------------------------
// Persistent CTAs (one per SM).  A work unit is 256 rows = two 128-row tiles that share every weight stage, times ALL
// N <= 256 output columns: the two fp32 accumulators fill the TMEM.  Warp roles: 0-7 load the fp32 rows and split
// them (three K = 16 steps in flight per thread), 8 and 14 issue the MMAs (one tile each), 9 streams the split weights
// with bulk copies, 10-13 are the epilogue (bias from shared memory, ReLU / ReLU' mask, fp32 rows to HBM) -- while
// they drain a unit the loads, splits and bulk copies of the next one already fill the stage ring.
// What the measurements said (profiles/r02_fp32_tc.md): the kernel is bound by its LOAD / STORE PATH, not by the
// tensor pipe -- removing every MMA but one changed the time by 5 %, removing the A loads by 34 %, the C stores by
// 19 %.  Hence: A is read once per unit (column-block units re-read it: slower although their epilogue overlapped
// the next unit's MMAs), a load instruction covers 8 rows x 64 contiguous bytes instead of 32 rows x 16, the bias
// comes from shared memory (per-element global loads were 37 % of all stall samples), and 128-row CTAs (two per SM)
// lost to the 6-byte-per-element weight stream they each had to re-fetch.
constexpr int kGThreads = 480;          // warps 0-7 split A, 8 and 14 = MMA issue (tile 0 / tile 1), 9 = bulk copies,
                                        // 10-13 = epilogue
constexpr int kGStages = 4;
struct GemmSmem {
  // per stage: A [2 tiles][3 splits][2 chunks][128 rows][8] = 24 KB, B [3][2][N <= 256][8] = 24 KB
  uint8_t a[kGStages][2 * 3 * 4096];
  uint8_t b[kGStages][3 * 8192];
  float bias[256];                      // staged once: a scalar global load per column and row sat on the epilogue's
                                        // critical path (ncu: 37 % of all stall samples on the dependent FADDs)
  uint64_t full[kGStages], a_ready[kGStages], empty[kGStages], acc_ready, acc_free;
  uint32_t tmem_base;
};

struct XGemmArgs {
  const float* A1; int lda1; int K1; const uint8_t* B1;
  const float* A2; int lda2; int K2; const uint8_t* B2;
  const float* bias; float* C; int ldc; int64_t M; int N; int epi;
  const float* mask; int ldmask;
};

__global__ void __launch_bounds__(kGThreads, 1) tcx_gemm_kernel(XGemmArgs g) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  GemmSmem& sm = *reinterpret_cast<GemmSmem*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = g.N;
  const int ks1 = (g.K1 + 15) / 16, ks2 = (g.K2 + 15) / 16, ksteps = ks1 + ks2;
  const int64_t n_units = (g.M + 255) / 256;                  // unit = 256-row block
  const int64_t first = blockIdx.x, stride = gridDim.x;
  if (tid == 0) {
    // empty / acc_ready: one tcgen05.commit from EACH of the two issuing threads
    for (int i = 0; i < kGStages; ++i) { mbar_init(&sm.full[i], 1); mbar_init(&sm.a_ready[i], 8); mbar_init(&sm.empty[i], 2); }
    mbar_init(&sm.acc_ready, 2); mbar_init(&sm.acc_free, 4);
    fence_mbar_init();
  }
  if (warp == 8) tmem_alloc<512>(&sm.tmem_base);
  for (int i = tid; i < N; i += kGThreads) sm.bias[i] = g.bias != nullptr ? __ldg(g.bias + i) : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sm.tmem_base;
  const uint32_t stage_bytes = 96u * (uint32_t)N;

  if (warp == 9) {
    // ---- weight-operand producer: one bulk copy per (unit, K = 16 step) ----
    if (lane == 0) {
      uint32_t it = 0;
      for (int64_t u = first; u < n_units; u += stride) {
        for (int kt = 0; kt < ksteps; ++kt, ++it) {
          const uint32_t s = it % kGStages;
          if (it >= (uint32_t)kGStages) mbar_wait(&sm.empty[s], ((it / kGStages) - 1) & 1);
          const uint8_t* src = (kt < ks1) ? g.B1 + (size_t)kt * stage_bytes : g.B2 + (size_t)(kt - ks1) * stage_bytes;
          mbar_arrive_expect_tx(&sm.full[s], stage_bytes);
          tma_load_1d(sm.b[s], src, stage_bytes, &sm.full[s]);
        }
      }
    }
  } else if (warp == 8 || warp == 14) {
    // ---- MMA issuers: per step six bf16 x bf16 products into the fp32 accumulator of THIS thread's tile.  Two
    //      threads because tcgen05.mma holds its issuer for ~160 cycles per N = 128 MMA whose pipe time is 64
    //      (DESIGN.md §4 note 10): one thread alone ran the pipe at 40 %.  Each accumulator has ONE issuer, so the
    //      fp32 summation order -- every output bit -- is fixed ----
    if (lane == 0) {
      const int tile = warp == 8 ? 0 : 1;
      const uint32_t idesc = umma_idesc_bf16(128, N, 0, 0);
      uint32_t it = 0, un = 0;
      for (int64_t u = first; u < n_units; u += stride, ++un) {
        if (un >= 1) {   // the epilogue warps have drained the previous unit (the accumulators fill the TMEM)
          mbar_wait(&sm.acc_free, (un - 1) & 1);
          tc_fence_after();
        }
        for (int kt = 0; kt < ksteps; ++kt, ++it) {
          const uint32_t s = it % kGStages, ph = (it / kGStages) & 1;
          mbar_wait(&sm.full[s], ph);
          mbar_wait(&sm.a_ready[s], ph);
          tc_fence_after();
          const uint32_t a0 = smem_u32(sm.a[s]), b0 = smem_u32(sm.b[s]);
#pragma unroll
          for (int p = 0; p < 6; ++p) {
            const uint64_t da = umma_smem_desc(a0 + tile * 12288 + kProdA[p] * 4096, 2048, 128);
            const uint64_t db = umma_smem_desc(b0 + kProdB[p] * 32 * N, 16 * N, 128);
            umma_bf16(tmem + tile * 256, da, db, idesc, (kt > 0 || p > 0) ? 1u : 0u);
          }
          umma_commit(&sm.empty[s]);
        }
        umma_commit(&sm.acc_ready);
      }
    }
  } else if (warp < 8) {
    // ---- A-split warps: warp w owns rows 32 w .. 32 w + 31 of the 256-row unit (tile w >> 2).  One load instruction
    //      covers 8 rows x 64 contiguous bytes (lane = (row & 7) * 4 + quarter): 8 lines / 16 fully used sectors per
    //      request.  (One row per lane -- 32 lines, half-used sectors per request -- ran the loop at the L1 tag rate:
    //      ncu showed these warps waiting on their loads although three steps were in flight.)  The quarter's four
    //      values become 8 bytes of each split operand: a warp's store is two contiguous 128-byte runs (conflict
    //      free).  Three steps are kept in flight in a register ring (compile-time index in the 4x unrolled body). ----
    const int tile = warp >> 2, r8 = lane >> 2, qk = lane & 3;
    const int row0 = (warp & 3) * 32 + r8;                      // + 8 j, j = 0..3
    int64_t n_mine = 0;
    for (int64_t u = first; u < n_units; u += stride) ++n_mine;
    const int64_t total = n_mine * ksteps;
    auto fetch = [&](int64_t gi, float4 (&x)[4]) {
      const int64_t un = gi / ksteps;
      const int kt = (int)(gi - un * ksteps);
      const int64_t grow = (first + un * stride) * 256 + tile * 128 + row0;
      const bool second = kt >= ks1;
      const float* A = second ? g.A2 : g.A1;
      const int lda = second ? g.lda2 : g.lda1, K = second ? g.K2 : g.K1, k0 = (second ? kt - ks1 : kt) * 16 + qk * 4;
#pragma unroll
      for (int j = 0; j < 4; ++j) x[j] = load_a4(A, lda, K, grow + 8 * j, g.M, k0);
    };
    float4 xr[4][4];
#pragma unroll
    for (int u = 0; u < 3; ++u)
      if (u < total) fetch(u, xr[u]);
    for (int64_t g0 = 0; g0 < total; g0 += 4) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int64_t gi = g0 + u;
        if (gi < total) {
          if (gi + 3 < total) fetch(gi + 3, xr[(u + 3) & 3]);
          uint2 p1[4], p2[4], p3[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) split3x4(xr[u][j], p1[j], p2[j], p3[j]);
          const uint32_t it = (uint32_t)gi, s = it % kGStages;
          if (it >= (uint32_t)kGStages) mbar_wait(&sm.empty[s], ((it / kGStages) - 1) & 1);
          // chunk (qk >> 1) of the step, row row0 + 8 j, half (qk & 1) of the 16-byte vector
          uint8_t* dst = sm.a[s] + tile * 12288 + (qk >> 1) * 2048 + row0 * 16 + (qk & 1) * 8;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            *reinterpret_cast<uint2*>(dst + j * 128) = p1[j];
            *reinterpret_cast<uint2*>(dst + j * 128 + 4096) = p2[j];
            *reinterpret_cast<uint2*>(dst + j * 128 + 8192) = p3[j];
          }
          fence_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(&sm.a_ready[s]);
        }
      }
    }
  } else {
    // ---- epilogue warps 10..13: TMEM lane quadrant = warp & 3; both tiles, all N columns of the unit ----
    const int q = warp & 3;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    uint32_t un = 0;
    for (int64_t u = first; u < n_units; u += stride, ++un) {
      mbar_wait(&sm.acc_ready, un & 1);
      tc_fence_after();
#pragma unroll 1
      for (int tl = 0; tl < 2; ++tl) {
        const int64_t orow = u * 256 + tl * 128 + q * 32 + lane;
        const bool live = orow < g.M;
        for (int col = 0; col < N; col += 32) {
          uint32_t v[32];
          tmem_ld32_issue(tmem + lane_base + tl * 256 + col, v);   // warp-collective: outside the row guard
          // the ReLU' mask row (dgrad) is fetched while the TMEM load is in flight
          float4 mk[8];
          if (g.epi == 3 && live) {
#pragma unroll
            for (int i = 0; i < 8; ++i) mk[i] = __ldg(reinterpret_cast<const float4*>(g.mask + orow * g.ldmask + col) + i);
          }
          tmem_ld32_wait(v);
          if (live) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 bb = *reinterpret_cast<const float4*>(&sm.bias[col + 4 * i]);
              float4 o = make_float4(__uint_as_float(v[4 * i]) + bb.x, __uint_as_float(v[4 * i + 1]) + bb.y,
                                     __uint_as_float(v[4 * i + 2]) + bb.z, __uint_as_float(v[4 * i + 3]) + bb.w);
              if (g.epi == 1) {          // EPI_RELU
                o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f);
              } else if (g.epi == 3) {   // EPI_MASK: C = acc * (mask > 0)
                o.x = mk[i].x > 0.f ? o.x : 0.f; o.y = mk[i].y > 0.f ? o.y : 0.f;
                o.z = mk[i].z > 0.f ? o.z : 0.f; o.w = mk[i].w > 0.f ? o.w : 0.f;
              }
              *reinterpret_cast<float4*>(g.C + orow * g.ldc + col + 4 * i) = o;
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&sm.acc_free);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) tmem_dealloc<512>(tmem);
}

// ---- dW[K,N] += A[M,K]^T Z[M,N] -------------------------------------------------------------------------------
constexpr int kWSamples = 32;           // samples per stage (two K = 16 MMA steps)
constexpr int kWStages = 2;
struct WgSmem {
  // per stage: A [3 splits][32 feature chunks][32 samples][8] = 48 KB, Z likewise ([N/8 chunks])
  uint8_t a[kWStages][3 * 16384];
  uint8_t z[kWStages][3 * 16384];
  uint64_t ready[kWStages], empty[kWStages], acc_ready;
  uint32_t tmem_base;
};

__global__ void __launch_bounds__(kXThreads, 1)
tcx_wgrad_kernel(const float* __restrict__ A, int lda, int K, const float* __restrict__ Z, int ldz, int N, int64_t M,
                 int64_t slab, float* __restrict__ dW, int ldw, float* __restrict__ db) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  WgSmem& sm = *reinterpret_cast<WgSmem*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t mb = (int64_t)blockIdx.x * slab, me = min(mb + slab, M);
  const int nst = (int)((me - mb + kWSamples - 1) / kWSamples);
  const int halves = (K + 127) / 128;                // 128-row accumulator blocks (TMEM columns h * 256)
  if (tid == 0) {
    for (int i = 0; i < kWStages; ++i) { mbar_init(&sm.ready[i], 8); mbar_init(&sm.empty[i], 2); }
    mbar_init(&sm.acc_ready, 2);
    fence_mbar_init();
  }
  if (warp == 8) tmem_alloc<512>(&sm.tmem_base);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sm.tmem_base;

  if (warp >= 8) {
    // two issuing threads, one per 128-row accumulator block h (a single thread runs the pipe at ~2/3: tcgen05.mma
    // holds its issuer); with K <= 128 the second one only keeps the barrier counts
    if (lane == 0 && nst > 0) {
      const int h = warp - 8;
      const uint32_t idesc = umma_idesc_bf16(128, N, 1, 1);
      for (int st = 0; st < nst; ++st) {
        const int s = st % kWStages;
        mbar_wait(&sm.ready[s], (st / kWStages) & 1);
        tc_fence_after();
        const uint32_t a0 = smem_u32(sm.a[s]), z0 = smem_u32(sm.z[s]);
        if (h < halves) {
#pragma unroll
          for (int p = 0; p < 6; ++p) {
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {   // MN-major: LBO = 128 B (next 8 samples), SBO = 512 B (next 8 features)
              const uint64_t da = umma_smem_desc(a0 + kProdA[p] * 16384 + h * 8192 + ks * 256, 128, 512);
              const uint64_t dz = umma_smem_desc(z0 + kProdB[p] * 16384 + ks * 256, 128, 512);
              umma_bf16(tmem + h * 256, da, dz, idesc, (st > 0 || p > 0 || ks > 0) ? 1u : 0u);
            }
          }
          umma_commit(&sm.empty[s]);
        } else {
          mbar_arrive(&sm.empty[s]);
        }
      }
      if (h < halves) umma_commit(&sm.acc_ready);
      else mbar_arrive(&sm.acc_ready);
    }
  } else if (warp < 8) {
    // ---- compute warps: one load instruction covers 8 samples x 64 contiguous bytes (lane = (sample & 7) * 4 +
    //      quarter; the quarter's 4 features are 8 bytes of each split operand), groups of 16 features are dealt
    //      round-robin to the warps; all of a stage's loads are issued before the first is used ----
    const int s8 = lane >> 2, qk = lane & 3;
    const int ga = 8 * halves, gz = N / 16;            // 16-feature groups of A (zero-filled to 128 rows) and Z
    // bias gradient (db != nullptr): column sums of Z -- this thread sees, for its two feature groups, 4 features of
    // every 8th sample of the slab; partial sums stay in registers, one shuffle reduction + atomics at the end
    float4 bsum[2] = {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)};
    // (prefetching the next stage's loads into a second register set was tried: 128 more live registers, spills,
    // 14.8 -> 22.1 ms for the backward -- the two shared-memory stages already overlap a stage's loads with the
    // previous stage's MMAs)
    for (int st = 0; st < nst; ++st) {
      const int s = st % kWStages;
      const int64_t r0 = mb + (int64_t)st * kWSamples + s8;
      float4 xa[2][4], xz[2][4];
#pragma unroll
      for (int gi = 0; gi < 2; ++gi) {
        const int ga_i = warp + 8 * gi;
#pragma unroll
        for (int sb = 0; sb < 4; ++sb) {
          const int64_t r = r0 + 8 * sb;
          if (ga_i < ga) xa[gi][sb] = load_a4(A, lda, K, r < me ? r : M, M, ga_i * 16 + qk * 4);
          if (ga_i < gz) xz[gi][sb] = load_a4(Z, ldz, N, r < me ? r : M, M, ga_i * 16 + qk * 4);
        }
      }
      if (st >= kWStages) mbar_wait(&sm.empty[s], ((st / kWStages) - 1) & 1);
#pragma unroll
      for (int gi = 0; gi < 2; ++gi) {
        const int g_i = warp + 8 * gi;
        // chunk 2 g + (qk >> 1), sample s8 + 8 sb, half (qk & 1) of the 16-byte vector
        const int off = (2 * g_i + (qk >> 1)) * 512 + s8 * 16 + (qk & 1) * 8;
#pragma unroll
        for (int sb = 0; sb < 4; ++sb) {
          uint2 p1, p2, p3;
          if (g_i < ga) {
            split3x4(xa[gi][sb], p1, p2, p3);
            uint8_t* d = sm.a[s] + off + sb * 128;
            *reinterpret_cast<uint2*>(d) = p1;
            *reinterpret_cast<uint2*>(d + 16384) = p2;
            *reinterpret_cast<uint2*>(d + 32768) = p3;
          }
          if (g_i < gz) {
            bsum[gi].x += xz[gi][sb].x; bsum[gi].y += xz[gi][sb].y; bsum[gi].z += xz[gi][sb].z; bsum[gi].w += xz[gi][sb].w;
            split3x4(xz[gi][sb], p1, p2, p3);
            uint8_t* d = sm.z[s] + off + sb * 128;
            *reinterpret_cast<uint2*>(d) = p1;
            *reinterpret_cast<uint2*>(d + 16384) = p2;
            *reinterpret_cast<uint2*>(d + 32768) = p3;
          }
        }
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&sm.ready[s]);
    }
    if (db != nullptr) {
#pragma unroll
      for (int gi = 0; gi < 2; ++gi) {
        float v[4] = {bsum[gi].x, bsum[gi].y, bsum[gi].z, bsum[gi].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {       // lanes with the same quarter (lane & 3) hold the other samples
          v[e] += __shfl_xor_sync(0xffffffffu, v[e], 4);
          v[e] += __shfl_xor_sync(0xffffffffu, v[e], 8);
          v[e] += __shfl_xor_sync(0xffffffffu, v[e], 16);
        }
        const int g_i = warp + 8 * gi;
        if (s8 == 0 && g_i < gz && nst > 0) {
#pragma unroll
          for (int e = 0; e < 4; ++e) atomicAdd(db + g_i * 16 + qk * 4 + e, v[e]);
        }
      }
    }
    if (nst > 0) {
      mbar_wait(&sm.acc_ready, 0);
      tc_fence_after();
      const int q = warp & 3, hcol = warp >> 2;
      const uint32_t lane_base = (uint32_t)(q * 32) << 16;
      for (int h = 0; h < halves; ++h) {
        const int krow = h * 128 + q * 32 + lane;
        for (int c0 = hcol * (N / 2); c0 < (hcol + 1) * (N / 2); c0 += 32) {
          float v[32];
          tmem_ld32(tmem + lane_base + h * 256 + c0, v);
          if (krow < K) {
            float* dst = dW + (int64_t)krow * ldw + c0;
#pragma unroll
            for (int i = 0; i < 32; ++i) atomicAdd(dst + i, v[i]);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) tmem_dealloc<512>(tmem);
}

}  // namespace

// ---- host side ------------------------------------------------------------------------------------------------
size_t tcx_blob_bytes(int N, int K) { return (size_t)((K + 15) / 16) * 96 * N; }

int tcx_pack(const float* src, int ld, int N, int K, bool trans, void* blob, cudaStream_t st) {
  const int total = ((K + 15) / 16) * 2 * N;
  if (total == 0) return KNERF_OK;
  tcx_pack_kernel<<<std::min((total + 255) / 256, kNumSMs * 4), 256, 0, st>>>(src, ld, N, K, trans ? 1 : 0, (uint8_t*)blob);
  KN_LAUNCH_CHECK();
  return KNERF_OK;
}

// shapes the tensor kernels take: N a multiple of 64 up to 256, 16-byte aligned rows of C / bias / mask
bool tcx_gemm_eligible(const GemmArgs& g) {
  return g.N >= 64 && g.N <= 256 && g.N % 64 == 0 && (g.ldc & 3) == 0 && (g.K1 + g.K2) >= 16 &&
         (g.epi == EPI_NONE || g.epi == EPI_RELU || (g.epi == EPI_MASK && (g.ldmask & 3) == 0)) &&
         (reinterpret_cast<uintptr_t>(g.C) & 15) == 0 &&
         (g.epi != EPI_MASK || (reinterpret_cast<uintptr_t>(g.mask) & 15) == 0);
}

int launch_gemm_tc(const GemmArgs& g, const void* blob1, const void* blob2, cudaStream_t st) {
  if (g.M == 0) return KNERF_OK;
  XGemmArgs x{g.A1, g.lda1, g.K1, (const uint8_t*)blob1, g.A2, g.lda2, g.K2, (const uint8_t*)blob2,
              g.bias, g.C, g.ldc, g.M, g.N, g.epi, g.mask, g.ldmask};
  if (x.A1 == nullptr) x.K1 = 0;
  if (x.A2 == nullptr) x.K2 = 0;
  const size_t smem = sizeof(GemmSmem);
  KN_CUDA(cudaFuncSetAttribute(tcx_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  tcx_gemm_kernel<<<(unsigned)std::min<int64_t>(cdiv(g.M, 256), kNumSMs), kGThreads, smem, st>>>(x);
  KN_LAUNCH_CHECK();
  return KNERF_OK;
}

bool tcx_wgrad_eligible(int K, int N) { return K >= 16 && K <= 256 && N >= 64 && N <= 256 && N % 64 == 0; }

int launch_wgrad_tc(const float* A, int lda, int K, const float* Z, int ldz, int N, int64_t M, float* dW, int ldw,
                    float* db, cudaStream_t st) {
  if (M == 0) return KNERF_OK;
  const int64_t stages = cdiv(M, kWSamples);
  const int grid = (int)std::min<int64_t>(kNumSMs, stages);
  const int64_t slab = cdiv(stages, grid) * kWSamples;
  const size_t smem = sizeof(WgSmem);
  KN_CUDA(cudaFuncSetAttribute(tcx_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  tcx_wgrad_kernel<<<(unsigned)cdiv(M, slab), kXThreads, smem, st>>>(A, lda, K, Z, ldz, N, M, slab, dW, ldw, db);
  KN_LAUNCH_CHECK();
  return KNERF_OK;
}

}  // namespace knerf
