// Pieces shared by the fused forward and dgrad "chain" kernels (tc_roles2.cuh has the TMA producer and the
// tcgen05.mma issuers): optional in-kernel cycle counters and the record-store warp.  A chain kernel walks
// Prog::kSteps GEMM steps for two 128-sample tiles per CTA in ping-pong; the compute warps (kernel specific) turn
// each accumulator into the next step's A operand.
#pragma once

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
#else
#define KN_PROF_DECL()
#define KN_PROF_BEGIN(var)
#define KN_PROF_END(var, slot)
#define KN_PROF_FLUSH()
#endif

// warp 10, one lane (training kernels): every operand tile the compute warps leave in hs[tl] is also a saved
// record -- written to HBM by bulk copies instead of 16 STG.128 per compute thread.  Protocol per tile slot:
// compute warps arrive on st_ready[tl] (one arrive per warp) once their part of hs[tl] is written and fenced;
// this thread stores the tile, waits until the copy engine has read shared memory and arrives on st_done[tl],
// which the compute warps wait for before they overwrite hs[tl] in their next epilogue.
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

// compute warps, after their writes to hs[tl] are fenced (fence.proxy.async) and the warp has converged
__device__ __forceinline__ void st_ready_arrive(uint64_t* bar, int lane) {
  if (lane == 0) mbar_arrive(bar);
}

}  // namespace tcl
}  // namespace knerf
