// Blackwell (sm_100a) PTX wrappers used by the tcgen05 MLP kernels: mbarrier, TMA bulk copies,
// TMEM allocation, tcgen05.mma / .ld / .commit, UMMA shared-memory and instruction descriptors.
//
// Operand layout convention used everywhere in this library ("chunk-major", UMMA LayoutType SWIZZLE_NONE):
// a [rows x K] bf16 operand is stored as  [K/8 chunks][rows][8 elements]  -- one 16-byte vector per
// (chunk, row).  For a K-major operand (A = activations [samples x features], B = weights [out x in]) this
// is the canonical interleaved layout ((8,m),(T,2)):((1T,SBO),(1,LBO)) with
//     SBO = 128 B        (8 consecutive rows = one 128-byte core matrix, row groups are contiguous)
//     LBO = rows * 16 B  (next 8-element K chunk)
// and the SAME bytes read along the other axis are the canonical MN-major layout
// ((T,1,m),(8,k)):((1,T,SBO),(1T,LBO)) with  LBO = 128 B (next 8 k),  SBO = rows * 16 B (next 8 m|n),
// which is how the weight-gradient GEMM (reduction over samples) consumes the saved activations.
// A warp that owns 32 consecutive rows writes 512 contiguous bytes per chunk: no bank conflicts, no swizzle.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

namespace knerf {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {}
}

// ---- proxies / fences ----------------------------------------------------------------------------------
// generic-proxy smem writes -> visible to the async proxy (tcgen05.mma operand reads, bulk stores)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- TMA: 1-D bulk copies (UBLKCP) -----------------------------------------------------------------------
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// L2 eviction policies: the packed weights are re-read by every CTA for every tile (keep: evict_last) while the
// saved records stream through once (evict_first), otherwise the record writes push the weights out of L2
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void tma_load_1d_hint(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar,
                                                 uint64_t policy) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
               ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy) : "memory");
}

// smem -> global bulk store (bulk async-group completion): one thread moves a whole operand tile
__device__ __forceinline__ void tma_store_1d(void* gmem_dst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
               ::"l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_store_1d_hint(void* gmem_dst, const void* smem_src, uint32_t bytes, uint64_t policy) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
               ::"l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes), "l"(policy) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all bulk stores of this thread have finished READING shared memory (the source may be overwritten)
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// ... all but the most recent group
__device__ __forceinline__ void tma_store_wait_read_1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }

// ---- TMEM ----------------------------------------------------------------------------------------------
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result) {   // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "n"(COLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t addr) {         // the same warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "n"(COLS) : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread = lane (row), register i = column base+i.
// Split form: issue the asynchronous load, do independent work (prefetch the next bias / mask vectors), then
// wait.  The wait lists the destination registers as read-write operands so that no use can be scheduled
// above it.
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld32_wait(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                 "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                 "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :: "memory");
}

// 8 consecutive columns (the forward's last step: the head pre-activations as hi + lo parts)
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// ---- UMMA descriptors ------------------------------------------------------------------------------------
// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46)
// | version=1 [46,48) | base_offset [49,52) | lbo_mode [52] | layout_type [61,64) (0 = SWIZZLE_NONE)
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}

// instruction descriptor (cute::UMMA::InstrDescriptor), kind::f16, bf16 x bf16 -> fp32:
// c_format=F32 [4,6) | a_format=BF16 [7,10) | b_format=BF16 [10,13) | a_major [15] | b_major [16] (0 = K, 1 = MN)
// | N>>3 [17,23) | M>>4 [24,29)
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread for the whole CTA
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}

// kind::f8f6f4, fp8 x fp8 -> fp32 (K = 32 per instruction): same descriptor fields, a_format / b_format 0 = E4M3,
// 1 = E5M2 (cute::UMMA::InstrDescriptor).  8-bit operands may be MN-major too; the chunk-major layout becomes
// [rows/16 chunks][K][16 elements] -- still one 16-byte vector per (chunk, k), LBO = 128 B (next 8 k), SBO = K * 16 B.
constexpr int kE4M3 = 0, kE5M2 = 1;
__host__ __device__ constexpr uint32_t umma_idesc_f8(int M, int N, int a_fmt, int b_fmt, int a_mn_major, int b_mn_major) {
  return (1u << 4) | ((uint32_t)a_fmt << 7) | ((uint32_t)b_fmt << 10) | ((uint32_t)a_mn_major << 15) |
         ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_f8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}

// arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed
// (implies tcgen05.fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// p[0..3] += (a, b, c, d) in global memory as ONE 16-byte reduction (REDG.E.ADD.F32x4); p must be 16-byte aligned
__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// ---- small numeric helpers -------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
// max(.,0) fused into the conversion (F2FP.RELU.BF16.F32.PACK_AB): low half = lo, high half = hi
__device__ __forceinline__ uint32_t pack_bf16x2_relu(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
// four fp32 -> four fp8 bytes (byte i = value i), round to nearest, saturating to the largest finite value
__device__ __forceinline__ uint32_t pack_e4m3x4_relu(float a, float b, float c, float d) {
  uint32_t r;
  asm("{\n\t.reg .b16 lo, hi;\n\t"
      "cvt.rn.satfinite.relu.e4m3x2.f32 lo, %2, %1;\n\t"
      "cvt.rn.satfinite.relu.e4m3x2.f32 hi, %4, %3;\n\t"
      "mov.b32 %0, {lo, hi};\n\t}"
      : "=r"(r) : "f"(a), "f"(b), "f"(c), "f"(d));
  return r;
}
__device__ __forceinline__ uint32_t pack_e4m3x4(float a, float b, float c, float d) {
  uint32_t r;
  asm("{\n\t.reg .b16 lo, hi;\n\t"
      "cvt.rn.satfinite.e4m3x2.f32 lo, %2, %1;\n\t"
      "cvt.rn.satfinite.e4m3x2.f32 hi, %4, %3;\n\t"
      "mov.b32 %0, {lo, hi};\n\t}"
      : "=r"(r) : "f"(a), "f"(b), "f"(c), "f"(d));
  return r;
}
__device__ __forceinline__ uint32_t pack_e5m2x4(float a, float b, float c, float d) {
  uint32_t r;
  asm("{\n\t.reg .b16 lo, hi;\n\t"
      "cvt.rn.satfinite.e5m2x2.f32 lo, %2, %1;\n\t"
      "cvt.rn.satfinite.e5m2x2.f32 hi, %4, %3;\n\t"
      "mov.b32 %0, {lo, hi};\n\t}"
      : "=r"(r) : "f"(a), "f"(b), "f"(c), "f"(d));
  return r;
}
// acc += an fp16 value: one instruction (FHADD, which reads either half of a register), exact fp16 -> fp32 and one fp32
// rounding -- the same bits as a conversion followed by an fp32 add
__device__ __forceinline__ float add_f16(float acc, unsigned short h) {
  asm("add.rn.f32.f16 %0, %1, %0;" : "+f"(acc) : "h"(h));
  return acc;
}
// a[0..3] += the four e5m2 bytes of w.  An e5m2 byte is the upper byte of the fp16 with the same value, so one prmt
// makes two fp16 of two bytes.
__device__ __forceinline__ void add_e5m2x4(float* a, uint32_t w) {
  const uint32_t lo = __byte_perm(w, 0u, 0x1404), hi = __byte_perm(w, 0u, 0x3424);
  a[0] = add_f16(a[0], (unsigned short)(lo & 0xffffu)); a[1] = add_f16(a[1], (unsigned short)(lo >> 16));
  a[2] = add_f16(a[2], (unsigned short)(hi & 0xffffu)); a[3] = add_f16(a[3], (unsigned short)(hi >> 16));
}
// prmt.b32 in its default mode: a selector nibble with bit 3 set yields the SIGN of the selected byte replicated over
// the byte (0x00 / 0xff) -- one instruction turns flag bits parked in byte msbs into byte / half-word masks
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}
__device__ __forceinline__ float bf16_lo(uint32_t p) { return __uint_as_float(p << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t p) { return __uint_as_float(p & 0xffff0000u); }

}  // namespace tc
}  // namespace knerf

// ---- 2-CTA (cta_group::2) additions ------------------------------------------------------------------------
// A CTA pair (cluster of 2 on one TPC) executes ONE tcgen05.mma with M = 256: each CTA contributes its own 128
// rows of A and HALF of the B rows (N/2), so shared-memory operand traffic per SM is halved.
namespace knerf {
namespace tc {

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the mbarrier at the same shared-memory offset in CTA `cta` of the cluster.  Default semantics
// (.release.cta), as CUTLASS's ClusterBarrier::arrive(cta_id): the explicit .release.cluster form costs ~350
// cycles more per arrive (benchmarks/micro/umma_interf.cu) and sits on the epilogue -> MMA critical path.
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(smem_u32(bar)), "r"(cta) : "memory");
}
// wait on a local mbarrier that is (also) signalled from the peer CTA (remote arrive, multicast tcgen05.commit)
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) { mbar_wait(bar, parity); }

template <int COLS>
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* smem_result) {   // one full warp in EACH CTA of the pair
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "n"(COLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t addr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "n"(COLS) : "memory");
}

// D[tmem, both CTAs] (+)= A * B with M = 256; issued by ONE thread of the leader CTA
__device__ __forceinline__ void umma_bf16_2cta(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// completion of all prior MMAs -> arrive on the mbarrier at this offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}

}  // namespace tc
}  // namespace knerf
