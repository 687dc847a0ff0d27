// Roles of the fused forward and dgrad "chain" kernels.  A chain kernel walks Prog::kSteps GEMM steps; a CTA PAIR
// (cluster of 2 = one TPC) works on four 128-sample tiles -- two per CTA, ping-pong -- and every GEMM step is ONE
// M=256 tcgen05.mma per K=16 issued by the leader CTA: each CTA feeds its own A tile and HALF of the weight rows (N/2),
// so the shared-memory traffic per SM (operand reads + TMA writes) and the L2->SM weight traffic are both halved, which
// is what bounded the first, single-CTA version of these kernels (DESIGN.md §4).  Weight stages are K = 64 wide
// (tc_layout.cuh PairLayout): the issuing thread spends ~150 cycles per stage on barriers, so four MMAs (512 tensor
// cycles) per stage keep it ahead of the pipe where two (256 cycles) did not (benchmarks/micro/umma_rate.cu).
//
//   warp 0 lane 0 (both CTAs)  TMA producer: this CTA's piece of every weight stage, ONE bulk copy, 4-slot ring
//   warp 1 lane 0 (peer CTA)   relay: local "stage landed" -> arrive on the leader's full barrier of that slot
//   warps 1, 11 lane 0 (leader) MMA issuers; tcgen05.commit multicasts "slot free" / "accumulator ready" to both CTAs
//   warps 2-9    (both CTAs)   compute warps (kernel specific): turn each accumulator into the next step's A operand;
//                              "A operand ready" = one arrive per warp on the LEADER's barrier
//   warp 10 lane 0             record store (training kernels with bf16 records)
#pragma once

#include "common.cuh"
#include "tc_layout.cuh"
#include "tc_ptx.cuh"

namespace knerf {
namespace tcl {
using namespace tc;

// ---- optional in-kernel timing (build with -DKNERF_TC_TIMING; off by default, zero cost) ----------------------
// per CTA, clock64() cycles: slot 0 producer waits for a free stage | 1 MMA thread waits for the A operand |
// 2 MMA thread waits for a weight stage | 3 MMA thread total | 4 compute warp 2 waits for an accumulator |
// 5 compute total | 6.. per-step epilogue cycles of compute warp 2 (16 + s for tile slot 1) | 15, 31: the dgrad
// kernel's tile prologue (tile slot 0, 1)
#ifdef KNERF_TC_TIMING
static __device__ unsigned long long g_tc_prof[160][40];
// counters live in the thread's local memory (L1) and are flushed once at the end of the role
#define KN_PROF_DECL() unsigned long long kn_prof[40]; for (int kn_i = 0; kn_i < 40; ++kn_i) kn_prof[kn_i] = 0ull
#define KN_PROF_BEGIN(var) const long long var = clock64()
#define KN_PROF_END(var, slot) kn_prof[slot] += (unsigned long long)(clock64() - var)
// (atomic: both MMA issuers of a leader CTA flush into the same slots)
#define KN_PROF_FLUSH() for (int kn_i = 0; kn_i < 40; ++kn_i) if (kn_prof[kn_i]) atomicAdd(&g_tc_prof[blockIdx.x][kn_i], kn_prof[kn_i])
// host: copy up to n values of a per-CTA counter array (a __device__ symbol) to host_out and clear the array
template <class Counters>
int prof_read_and_clear(Counters& counters, unsigned long long* host_out, int n) {
  constexpr int kCount = (int)(sizeof(Counters) / sizeof(unsigned long long));
  static unsigned long long zeros[kCount];
  if (n > kCount) n = kCount;
  if (cudaMemcpyFromSymbol(host_out, counters, (size_t)n * 8) != cudaSuccess) return -1;
  if (cudaMemcpyToSymbol(counters, zeros, sizeof(zeros)) != cudaSuccess) return -1;
  return n;
}
#define KN_PROF_READ(counters, host_out, n) prof_read_and_clear(counters, host_out, n)
#else
#define KN_PROF_DECL()
#define KN_PROF_BEGIN(var)
#define KN_PROF_END(var, slot)
#define KN_PROF_FLUSH()
#define KN_PROF_READ(counters, host_out, n) ((void)(host_out), (void)(n), 0)
#endif

__device__ __forceinline__ uint32_t chain_setup(ChainSmem& sm, int tid, int warp, uint32_t cta) {
  if (tid == 0) {
    for (int i = 0; i < kNumStages; ++i) {
      // leader: its own producer (arrive + tx bytes) and the peer's relay; peer: its producer only
      mbar_init(&sm.full[i], cta == 0 ? 2 : 1);
      mbar_init(&sm.empty[i], 1);
    }
    sm.items_issued = 0u;
    sm.first_issued[0] = sm.first_issued[1] = 0u;
    for (int i = 0; i < 2; ++i) {
      mbar_init(&sm.a_ready[i], 16); mbar_init(&sm.acc_ready[i], 2);   // acc_ready: one commit per MMA issuer
      mbar_init(&sm.st_ready[i], 8); mbar_init(&sm.st_done[i], 1);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc_2cta<512>(&sm.tmem_base);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  return sm.tmem_base;
}

__device__ __forceinline__ void chain_teardown(uint32_t tmem, int warp) {
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc_2cta<512>(tmem);
}

// `blob` = the pair blob of this program (PairLayout<Prog>)
template <class Prog>
__device__ __forceinline__ void producer_role(ChainSmem& sm, const uint8_t* __restrict__ blob, uint32_t cta,
                                              int64_t n_quads, int64_t first, int64_t stride) {
  using PL = PairLayout<Prog>;
  uint32_t it = 0;
  const uint64_t pol = l2_policy_evict_last();
  KN_PROF_DECL();
  for (int64_t quad = first; quad < n_quads; quad += stride) {
#pragma unroll 1
    for (int s = 0; s < Prog::kSteps; ++s) {
      const int ns = PL::n_stages(s);
      const uint8_t* step_src = blob + PL::blob_off(s);
#pragma unroll 1
      for (int tl = 0; tl < 2; ++tl) {
#pragma unroll 1
        for (int i = 0; i < ns; ++i, ++it) {
          const uint32_t slot = it % kNumStages, ph = (it / kNumStages) & 1;
          const uint32_t pb = PL::piece_bytes(s, i);
          KN_PROF_BEGIN(t0);
          mbar_wait_cluster(&sm.empty[slot], ph ^ 1);
          KN_PROF_END(t0, 0);
          mbar_arrive_expect_tx(&sm.full[slot], pb);
          tma_load_1d_hint(sm.stage[slot], step_src + PL::stage_off(s, i) + cta * pb, pb, &sm.full[slot], pol);
        }
      }
    }
  }
  KN_PROF_FLUSH();
}

// peer CTA: forward "my piece of slot k has landed" to the leader's full barrier, in ring order
template <class Prog>
__device__ __forceinline__ void relay_role(ChainSmem& sm, int64_t n_quads, int64_t first, int64_t stride) {
  using PL = PairLayout<Prog>;
  uint32_t it = 0;
  for (int64_t quad = first; quad < n_quads; quad += stride) {
#pragma unroll 1
    for (int s = 0; s < Prog::kSteps; ++s) {
      const int n = PL::n_stages(s) * 2;
#pragma unroll 1
      for (int i = 0; i < n; ++i, ++it) {
        const uint32_t slot = it % kNumStages, ph = (it / kNumStages) & 1;
        mbar_wait(&sm.full[slot], ph);
        mbar_arrive_cluster(&sm.full[slot], 0);
      }
    }
  }
}

// TWO issuing threads (warps 1 and 11 of the leader CTA) take the ring items alternately: thread p issues the MMAs
// of the items with index % 2 == p.  tcgen05.mma holds its issuing thread until the MMA has (nearly) completed --
// measured: with one issuer every cycle it spends on barriers between two MMAs is a cycle the tensor pipe idles
// (benchmarks/micro/umma_rate.cu: stage time = MMA time + overhead, additive, ~250 cycles per stage).  With two
// issuers the pipe runs one thread's stage while the other waits for its next weight stage and commits.
//  * ring slot = item % 4, so every slot has exactly ONE consumer thread: the parity waits stay sound;
//  * both threads wait for a_ready[tl]; acc_ready[tl] expects one tcgen05.commit from each (a commit covers only
//    the MMAs of the committing thread);
//  * ordered = true (training kernels): the MMAs are ISSUED in ring order (items_issued, a counter in shared
//    memory: a thread issues item j once the other has issued item j-1), so the fp32 accumulation order -- hence
//    every output bit -- is the same as with a single issuer, run after run; the per-stage barrier work still
//    happens before that hand-over, off the pipe's critical path;
//  * ordered = false (inference): only the first MMA of a step (accumulate = 0, it overwrites the accumulator) is
//    ordered before the other thread's items of that step (first_issued[tl], a step counter).  The two threads'
//    later MMAs may interleave either way: sums of the same fp32 products in a different order, i.e. outputs
//    can differ in the last bit from run to run -- 16 % more throughput (1475 vs 1275 TFLOP/s).
// Accumulation into the same TMEM tile from two threads is safe: the pipe executes MMAs one at a time.
template <class Prog>
__device__ __forceinline__ void mma_role(ChainSmem& sm, uint32_t tmem, uint32_t p, bool ordered, int64_t n_quads,
                                         int64_t first, int64_t stride) {
  using PL = PairLayout<Prog>;
  uint32_t it = 0, a_par = 0;   // bit tl of a_par = parity of a_ready[tl]
  uint32_t step_no = 0;   // GEMM steps before the current one
  // descriptor templates: K-major SWIZZLE_NONE, SBO = 128 B, LBO = rows * 16 B; only the 14-bit start address varies
  const uint32_t stage0 = smem_u32(sm.stage[0]);
  KN_PROF_DECL();
  KN_PROF_BEGIN(t_all);
  for (int64_t quad = first; quad < n_quads; quad += stride) {
#pragma unroll 1
    for (int s = 0; s < Prog::kSteps; ++s) {
      const int nd = PL::n_data(s), kh = PL::kh(s);
      const int ns = PL::n_stages(s);
      const int N = Prog::N(s);
      const uint32_t idesc = umma_idesc_bf16(2 * kTileM, N, 0, 0);
      const uint32_t chunk_b = (uint32_t)N * 8;            // N/2 rows x 16 B
      const uint64_t db0 = umma_smem_desc(stage0, chunk_b, 128);
      const uint32_t db_step = (2 * chunk_b) >> 4;          // K = 16 further along a stage
#pragma unroll 1
      for (int tl = 0; tl < 2; ++tl) {
        const uint64_t da_hs = umma_smem_desc(smem_u32(sm.hs[tl]), kChunkA, 128);
        const uint64_t da_xs = umma_smem_desc(smem_u32(sm.xs[tl]), kChunkA, 128);
        const uint32_t d_tmem = tmem + tl * 256;
        volatile uint32_t* issued = &sm.items_issued;
        volatile uint32_t* fi = &sm.first_issued[tl];
        // Both threads wait for the A operand even when a step has only one item (dgrad step 0) and this thread none
        // of it: its acc_ready commit below must not arrive before the compute warps have taken the previous phase.
        KN_PROF_BEGIN(t_a);
        mbar_wait_cluster(&sm.a_ready[tl], (a_par >> tl) & 1);
        KN_PROF_END(t_a, 1);
        tc_fence_after();
        bool started = false;
#pragma unroll 1
        for (int i = 0; i < ns; ++i, ++it) {
          if ((it & 1u) != p) continue;
          if (!started) {   // this thread's first item of the step
            started = true;
            if (!ordered && i > 0) { while (*fi <= step_no) {} }   // item 0 (accumulate = 0) is the other thread's
          }
          const uint32_t slot = it % kNumStages, ph = (it / kNumStages) & 1;
          KN_PROF_BEGIN(t_f);
          mbar_wait_cluster(&sm.full[slot], ph);
          KN_PROF_END(t_f, 2);
          const uint64_t db = db0 + (uint64_t)(slot * (kStageBytes >> 4));
          if (ordered) { while (*issued != it) {} }         // my turn: every earlier item has been issued
          if (i < nd) {
            const int k0 = i * kPairK;
            const uint64_t da = (k0 < kh) ? da_hs + (uint64_t)((k0 >> 3) * (kChunkA >> 4))
                                          : da_xs + (uint64_t)(((k0 - kh) >> 3) * (kChunkA >> 4));
            const int nm = PL::stage_k(s, i) >> 4;          // 4, or 2 for the 32-wide tail
            umma_bf16_2cta(d_tmem, da, db, idesc, i > 0 ? 1u : 0u);
            if (!ordered && i == 0) *fi = step_no + 1;
            umma_bf16_2cta(d_tmem, da + 2 * (kChunkA >> 4), db + db_step, idesc, 1u);
            if (nm == 4) {
              umma_bf16_2cta(d_tmem, da + 4 * (kChunkA >> 4), db + 2 * db_step, idesc, 1u);
              umma_bf16_2cta(d_tmem, da + 6 * (kChunkA >> 4), db + 3 * db_step, idesc, 1u);
            }
          } else {   // + 1 * bias: A = the two encoding chunks holding the constant-1 column
            const uint64_t da = da_xs + (uint64_t)(Prog::bias_a_chunk(s) * (kChunkA >> 4));
            umma_bf16_2cta(d_tmem, da, db, idesc, 1u);
          }
          if (ordered) *issued = it + 1;
          umma_commit_2cta(&sm.empty[slot], 3);
        }
        a_par ^= 1u << tl;
        umma_commit_2cta(&sm.acc_ready[tl], 3);
      }
      ++step_no;
    }
  }
  KN_PROF_END(t_all, 3);
  KN_PROF_FLUSH();
}

// warp 10, one lane (training kernels with bf16 records): every operand tile the compute warps leave in hs[tl] is
// also a saved record -- written to HBM by bulk copies instead of 16 STG.128 per compute thread.  Protocol per tile
// slot: compute warps arrive on st_ready[tl] (one arrive per warp) once their part of hs[tl] is written and fenced;
// this thread stores the tile, waits until the copy engine has read shared memory and arrives on st_done[tl],
// which the compute warps wait for before they overwrite hs[tl] in their next epilogue (ChainHandshake).
// dst(item, tile) -> destination, bytes(item) -> size.
// The tile goes out in 16 KB pieces with at most two in flight: a whole-tile copy ahead of them in the SM's copy
// queue delays the weight stages (measured: the MMA thread then waits for stages a third of the time).
constexpr uint32_t kStorePiece = 16384;
template <class Smem, class TileOf, class Dst, class Bytes>
__device__ __forceinline__ void store_role(Smem& sm, int items_per_tile, int64_t n_tiles, int64_t n_units, int64_t first,
                                           int64_t stride, TileOf tile_of, Dst dst, Bytes bytes) {
  uint32_t par = 0;
  const uint64_t pol = l2_policy_evict_first();
  for (int64_t unit = first; unit < n_units; unit += stride) {
#pragma unroll 1
    for (int item = 0; item < items_per_tile; ++item) {
#pragma unroll 1
      for (int tl = 0; tl < 2; ++tl) {
        const int64_t tile = tile_of(unit, tl);
        mbar_wait(&sm.st_ready[tl], (par >> tl) & 1);
        par ^= 1u << tl;
        if (tile < n_tiles) {
          uint8_t* g = dst(item, tile);
          const uint32_t nb = bytes(item);
#pragma unroll 1
          for (uint32_t off = 0; off < nb; off += kStorePiece) {
            tma_store_1d_hint(g + off, sm.hs[tl] + off, kStorePiece, pol);
            tma_store_commit();
            tma_store_wait_read_1();
          }
          tma_store_wait_read();
        }
        mbar_arrive(&sm.st_done[tl]);
      }
    }
  }
}

// The compute warps' side of the hand-shakes, per tile slot tl.  STORE: the kernel has a store warp (store_role);
// without one (inference, fp8 records, which leave from the epilogue's registers) only the MMA hand-over remains.
template <bool STORE>
struct ChainHandshake {
  uint32_t pending = 0, par = 0;   // bit tl = hs[tl] is being stored / parity of st_done[tl]

  // this warp's part of the next A operand is written: publish it to the async proxy, then ONE arrive per warp on the
  // leader's barrier (16 = 8 warps x 2 CTAs); `record`: the tile in hs[tl] is also a saved record for the store warp
  __device__ __forceinline__ void arrive(ChainSmem& sm, int tl, int lane, bool record) {
    tc_fence_before();
    fence_async_smem();
    __syncwarp();
    if (lane == 0) mbar_arrive_cluster(&sm.a_ready[tl], 0);
    if (STORE && record) {
      if (lane == 0) mbar_arrive(&sm.st_ready[tl]);
      pending |= 1u << tl;
    }
  }
  // before the next write to hs[tl]: the bulk store of its previous contents has read them
  __device__ __forceinline__ void wait_writable(ChainSmem& sm, int tl) {
    if (STORE && ((pending >> tl) & 1)) {
      mbar_wait(&sm.st_done[tl], (par >> tl) & 1);
      par ^= 1u << tl;
      pending &= ~(1u << tl);
    }
  }
};

// host: launch a chain kernel as clusters of 2, at most one CTA pair per two SMs, each pair taking four tiles at a time
template <class... Params, class... Args>
int launch_chain(void (*kernel)(Params...), int64_t n_tiles, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cudaLaunchAttribute attr[1];
  cfg.blockDim = dim3(kThreads);
  cfg.stream = st;
  cfg.gridDim = dim3((unsigned)(2 * std::min<int64_t>(cdiv(n_tiles, 4), kNumSMs / 2)));
  cfg.dynamicSmemBytes = sizeof(ChainSmem);
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  KN_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cfg.dynamicSmemBytes));
  KN_CUDA(cudaLaunchKernelEx(&cfg, kernel, args...));
  KN_LAUNCH_CHECK();
  return KNERF_OK;
}

}  // namespace tcl
}  // namespace knerf
