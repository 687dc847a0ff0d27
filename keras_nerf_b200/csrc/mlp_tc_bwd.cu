// a11 (KNERF_BF16 mode): backward of the NeRF MLP on tcgen05 tensor cores.
//
//  1. tc_mlp_dgrad_kernel -- the forward's chain structure run backwards (same CTA-pair roles): starting from the
//     gradient w.r.t. the head pre-activations (from the fused compositing backward) it goes from (d rgb_pre, d sigma_pre)
//     straight to d(h7) through [W''' | w_s]^T (tc_layout.cuh: the heads are folded), then layer 7 .. layer 1, each step
//     one [128 x 256] x [256 x 256] GEMM followed by a ReLU' epilogue (1-bit masks written by the forward).
//     Every pre-activation gradient tile dZ_l is written once to HBM in chunk-major bf16 for step 2.
//     No gradient flows into the xyz / direction encodings (mlp.py inputs are constants: nerf.py:361-369).
//  2. tc_wgrad_kernel -- dW_l = X_l^T dZ_l with the reduction over SAMPLES: the saved activation / gradient
//     blobs are consumed as MN-major UMMA operands (same bytes, other axis; see tc_ptx.cuh), fp32 partial
//     sums stay in TMEM across all tiles of a work item and are flushed once with red.global.add.v4.f32; idle warps
//     take the bias gradients (column sums of the dZ units in shared memory).
//  3. tc_finish_kernel -- every gradient that contains d(rgb_features) = d(rgb_pre) Wc^T (rank 3): features,
//     rgb_features and rgb kernels / biases from Y = h7^T d(rgb_pre), Yd = PE(dir)^T d(rgb_pre), sum d(rgb_pre).
#include "mlp_tc.cuh"

#include <algorithm>
#include <cstdlib>
#include <vector>
#include "tc_roles.cuh"

namespace knerf {
using namespace tc;
using namespace tcl;

TcParams tc_make_params(const Model& m);

namespace {

// =============================================================================================================
// dgrad chain
// =============================================================================================================
// epilogue of one dgrad step: accumulator (dH = dZ_next W^T) -> pre-activation gradient tile, bf16.
// KIND 2: dZ_l = dH * ReLU'(h_l), l = 7..1;  3: dZ0, the last step: feeds no further GEMM, so it goes to HBM directly
// (dst = record or nullptr) and must NOT touch hs[tl], which the other half-row thread of this row may already be
// rebuilding for the next tile.  KIND < 3: dst = hs[tl], the next A operand and (via warp 10) the dZ record.
// mb = this thread's ReLU' bits (4 x 32 columns; bit 8 t + q = column 4 q + t of the group).
// REC8 (fp8 records): the dZ record leaves from here as e5m2(dZ * scale), 16 columns per 16-byte vector (rec8, nullptr
// for a padding tile); dst is only the next A operand then (unused for KIND 3).
template <int KIND, bool REC8>
__device__ __noinline__ void epi_dgrad(uint32_t tacc, uint8_t* __restrict__ dst, int h, int r, uint4 mbv,
                                       uint8_t* __restrict__ rec8) {
  const uint32_t mb[4] = {mbv.x, mbv.y, mbv.z, mbv.w};   // by value: no local memory (no L1 on this SM)
#pragma unroll
  for (int gI = 0; gI < 4; ++gI) {
    const int col0 = h * 128 + gI * 32;
    uint32_t v[32];
    tmem_ld32_issue(tacc + col0, v);
    tmem_ld32_wait(v);
    uint32_t q8[8];
#pragma unroll
    for (int c8 = 0; c8 < 4; ++c8) {
      float x[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) x[e] = __uint_as_float(v[c8 * 8 + e]);
      uint4 pk = make_uint4(pack_bf16x2(x[0], x[1]), pack_bf16x2(x[2], x[3]), pack_bf16x2(x[4], x[5]),
                            pack_bf16x2(x[6], x[7]));
      // ReLU' of columns 4q .. 4q+3 (q = 2 c8, 2 c8 + 1): bit q of bytes 0..3 of mb (tc_layout.cuh kRecMask).  Shifted left
      // by 7 - q they are the four byte msbs, and ONE prmt with sign replication expands two of them to a half-word
      // mask (the shift is an IMAD on the FMA pipe; the epilogue is bound by the half-rate ALU pipe)
      const uint32_t ta = mb[gI] << (7 - 2 * c8), tb = mb[gI] << (6 - 2 * c8);
      pk.x &= prmt(ta, 0u, 0x9988u); pk.y &= prmt(ta, 0u, 0xBBAAu);
      pk.z &= prmt(tb, 0u, 0x9988u); pk.w &= prmt(tb, 0u, 0xBBAAu);
      if (REC8) {   // byte masks of columns (0,1,2,3) / (4,5,6,7): the same flag bits of two words.  (The chain runs on
                    // gradients that already carry the record scale -- see the prologue -- so there is no multiply here.)
        q8[2 * c8] = pack_e5m2x4(x[0], x[1], x[2], x[3]) & prmt(ta, 0u, 0xBA98u);
        q8[2 * c8 + 1] = pack_e5m2x4(x[4], x[5], x[6], x[7]) & prmt(tb, 0u, 0xBA98u);
        if (KIND < 3) *reinterpret_cast<uint4*>(dst + ((col0 >> 3) + c8) * kChunkA + r * 16) = pk;
      } else {
        if (KIND < 3 || dst != nullptr) *reinterpret_cast<uint4*>(dst + ((col0 >> 3) + c8) * kChunkA + r * 16) = pk;
      }
    }
    if (REC8 && rec8 != nullptr) {
      __stcs(reinterpret_cast<uint4*>(rec8 + ((col0 >> 4) + 0) * kChunkA + r * 16), make_uint4(q8[0], q8[1], q8[2], q8[3]));
      __stcs(reinterpret_cast<uint4*>(rec8 + ((col0 >> 4) + 1) * kChunkA + r * 16), make_uint4(q8[4], q8[5], q8[6], q8[7]));
    }
  }
}

// fp8 records: max|d_pre| of the call (the bit pattern of a non-negative float orders like the float)
__global__ void __launch_bounds__(256) dpre_amax_kernel(const float4* __restrict__ d_pre, int64_t M,
                                                        uint32_t* __restrict__ amax_bits) {
  float m = 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < M; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = __ldg(d_pre + i);
    m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(amax_bits, __float_as_uint(m));
}

// clusters of 2, cta_group::2 MMAs (tc_roles.cuh); a work unit is four tiles (two per CTA)
template <bool REC8>
__global__ void __launch_bounds__(kThreads, 1)
tc_mlp_dgrad_kernel(const uint8_t* __restrict__ packed, const float4* __restrict__ d_pre, int64_t M,
                    const uint8_t* __restrict__ rec, uint8_t* __restrict__ dz, float* __restrict__ grads, TcParams P,
                    float* __restrict__ xbuf) {
  constexpr int kRB = REC8 ? kRec8Bytes : kRecBytes, kOffMask = REC8 ? kRec8Mask : kRecMask,
                kDB = REC8 ? kDz8Bytes : kDzBytes;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  ChainSmem& sm = *reinterpret_cast<ChainSmem*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t n_tiles = (M + kTileM - 1) / kTileM;
  const int64_t n_pairs = (n_tiles + 3) / 4;   // work units: four tiles per CTA pair
  const uint32_t cta = cluster_ctarank();
  const int64_t first = blockIdx.x >> 1, stride = gridDim.x >> 1;
  const uint32_t tmem = chain_setup(sm, tid, warp, cta);
  auto tile_of = [&](int64_t unit, int tl) -> int64_t { return unit * 4 + tl * 2 + (int64_t)cta; };

  if (warp == 0) {
    if (lane == 0) producer_role<BwdProg>(sm, packed + kBwdPairOff, cta, n_pairs, first, stride);
  } else if (warp == 1) {
    if (lane == 0 && cta == 0) mma_role<BwdProg>(sm, tmem, 0u, true, n_pairs, first, stride);
    else if (lane == 0) relay_role<BwdProg>(sm, n_pairs, first, stride);
  } else if (warp == 11) {
    if (lane == 0 && cta == 0) mma_role<BwdProg>(sm, tmem, 1u, true, n_pairs, first, stride);
  } else if (warp == 10) {
    // record store: the A operands dZ7..dZ1 of the chain (items 1..7) are also the dZ records of the weight-gradient
    // kernel (tc_roles.cuh store_role); item 0 = (d rgb_pre, d sigma_pre) only takes part in the hand-shake: the
    // prologue writes its record (kDzP)
    if (!REC8 && lane == 0) {   // (fp8 records leave from the epilogue's registers)
      store_role(sm, 8, n_tiles, n_pairs, first, stride, tile_of,
                 [&](int item, int64_t tile) {
                   return dz + tile * kDzBytes + (item == 0 ? kDzG : kDzZ0 + (8 - item) * kHSBytes);
                 },
                 [](int item) { return (uint32_t)(item == 0 ? 0 : kHSBytes); });   // dG stays on chip (item 0)
    }
  } else {
    ChainHandshake<!REC8> hk;   // (every A operand of the chain is also a dZ record)
    const int q = warp & 3, h = (warp - 2) >> 2;
    const int r = q * 32 + lane;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    uint32_t acc_par[2] = {0, 0};
    // fp8 records: one power-of-two scale per call, from max|d_pre| (written by dpre_amax_kernel before this launch)
    const float scale = REC8 ? dz8_scale(__ldg(reinterpret_cast<const uint32_t*>(xbuf) + kXOffAmax), false) : 1.f;

    KN_PROF_DECL();
    // tile start: (d rgb_pre, d sigma_pre, 0 ...) is the first A operand (K = 32, tc_layout.cuh BwdProg)
    auto prologue = [&](int64_t pair, int tl) {
      KN_PROF_BEGIN(t_p);
      const int64_t tile = tile_of(pair, tl);
      const int64_t g = tile * kTileM + r;
      const bool active = tile < n_tiles;
      float4 dp = make_float4(0.f, 0.f, 0.f, 0.f);
      if (g < M) dp = d_pre[g];
      // fp8 records: the whole chain runs on gradients times the record scale (a power of two: the same mantissas, so
      // every dZ is the same number times 2^k), and the e5m2 records need no multiply in the epilogues
      const float4 dq = REC8 ? make_float4(dp.x * scale, dp.y * scale, dp.z * scale, dp.w * scale) : dp;
      uint8_t* dz_t = dz + tile * kDB;
      const uint4 pk = (h == 0) ? make_uint4(pack_bf16x2(dq.x, dq.y), pack_bf16x2(dq.z, dq.w), 0u, 0u)
                                : make_uint4(0u, 0u, 0u, 0u);
      if (active && !REC8) *reinterpret_cast<uint4*>(dz_t + kDzP + h * kChunkA + r * 16) = pk;   // (dq = dp here)
      if (active && REC8 && h == 0)   // one 16-column chunk: (d rgb_pre, d sigma_pre) * scale, then zeros
        *reinterpret_cast<uint4*>(dz_t + kDz8P + r * 16) =
            make_uint4(pack_e5m2x4(dq.x, dq.y, dq.z, dq.w), 0u, 0u, 0u);
      if (h == 0) {   // bias gradients of the two heads: db_rgb = sum d(rgb_pre), db_sigma = sum d(sigma_pre)
        const float s0 = warp_sum(dp.x), s1 = warp_sum(dp.y), s2 = warp_sum(dp.z), s3 = warp_sum(dp.w);
        // sum d(rgb_pre) of THIS call for tc_finish_kernel, over the values the weight-gradient kernel's heads task
        // multiplies: the fp32 d_pre with fp8 records, the bf16 operand (kDzP) with bf16 records (dq = dp there)
        const float r0 = REC8 ? s0 : warp_sum(bf16_lo(pk.x)), r1 = REC8 ? s1 : warp_sum(bf16_hi(pk.x)),
                    r2 = REC8 ? s2 : warp_sum(bf16_lo(pk.y));
        if (lane == 0) {
          atomicAdd(grads + P.b_off[11], s0); atomicAdd(grads + P.b_off[11] + 1, s1);
          atomicAdd(grads + P.b_off[11] + 2, s2); atomicAdd(grads + P.b_off[8], s3);
          atomicAdd(xbuf + kXOffS, r0); atomicAdd(xbuf + kXOffS + 1, r1); atomicAdd(xbuf + kXOffS + 2, r2);
        }
      }
      hk.wait_writable(sm, tl);
      // chunk 0 of the row (h = 0), zeros in chunk 1 (h = 0) and chunks 2, 3 (h = 1): the step reads K = 32, and a
      // stale NaN pattern times a zero weight would not be zero
      *reinterpret_cast<uint4*>(sm.hs[tl] + (2 * h) * kChunkA + r * 16) = pk;
      *reinterpret_cast<uint4*>(sm.hs[tl] + (2 * h + 1) * kChunkA + r * 16) = make_uint4(0u, 0u, 0u, 0u);
      hk.arrive(sm, tl, lane, true);
      KN_PROF_END(t_p, 15 + tl * 16);
    };

    KN_PROF_BEGIN(t_c);
    if (first < n_pairs) {
#pragma unroll 1
      for (int tl = 0; tl < 2; ++tl) prologue(first, tl);
    }
    for (int64_t pair = first; pair < n_pairs; pair += stride) {
      for (int b = 0; b < BwdProg::kSteps; ++b) {
        const int zi = 7 - b;                                  // index of the dZ this step produces
#pragma unroll 1
        for (int tl = 0; tl < 2; ++tl) {
          const int64_t tile = tile_of(pair, tl);
          const bool active = tile < n_tiles;
          uint8_t* out = REC8 ? dz + tile * kDB + kDz8Z0 + zi * kH8Bytes : dz + tile * kDB + kDzZ0 + zi * kHSBytes;
          const uint8_t* mask = rec + tile * kRB + kOffMask + zi * kMaskLayerBytes;
          // the ReLU' bits (written by the forward, 1 bit per activation) do not depend on the accumulator: fetch
          // this thread's 4 x 32 columns BEFORE waiting for the MMA so that the latency overlaps it
          uint32_t mb[4] = {0u, 0u, 0u, 0u};
          if (active) {
            const uint4 mv = __ldg(reinterpret_cast<const uint4*>(mask + h * 2048 + r * 16));
            mb[0] = mv.x; mb[1] = mv.y; mb[2] = mv.z; mb[3] = mv.w;
          }
          KN_PROF_BEGIN(t_w);
          mbar_wait_cluster(&sm.acc_ready[tl], acc_par[tl]);
          KN_PROF_END(t_w, 4);
          KN_PROF_BEGIN(t_e);
          acc_par[tl] ^= 1;
          tc_fence_after();
          if (b + 1 < BwdProg::kSteps) hk.wait_writable(sm, tl);
          const uint32_t tacc = tmem + lane_base + tl * 256;
          const uint4 mbv = make_uint4(mb[0], mb[1], mb[2], mb[3]);
          uint8_t* out8 = (REC8 && active) ? out : nullptr;
          if (b + 1 < BwdProg::kSteps) epi_dgrad<2, REC8>(tacc, sm.hs[tl], h, r, mbv, out8);
          else epi_dgrad<3, REC8>(tacc, active ? out : nullptr, h, r, mbv, out8);
          if (b + 1 < BwdProg::kSteps) {
            hk.arrive(sm, tl, lane, true);
            KN_PROF_END(t_e, 6 + tl * 16 + b);
          } else {
            tc_fence_before();
            KN_PROF_END(t_e, 6 + tl * 16 + b);
            // (bias gradients = column sums of the dZ tiles are taken by tc_wgrad_kernel, which has them in smem)
            const int64_t next = pair + stride;
            if (next < n_pairs) prologue(next, tl);
          }
        }
      }
    }
    KN_PROF_END(t_c, 5);
    if (tid == 64) { KN_PROF_FLUSH(); }
  }
  chain_teardown(tmem, warp);
}

// =============================================================================================================
// weight gradients
// =============================================================================================================
constexpr int kWUnitBytes = 32768;     // 16 chunks x 128 samples x 16 B: 128 features (A) or 128 outputs (B)
constexpr int kWSlots = 7;            // 7 x 32 KB in flight per CTA (224 KB of the 227 KB)
constexpr int kWThreads = 224;         // warp 0 producer, warps 1 and 6 MMA issuers, warps 2-5 flush
constexpr int kNumTasks = 10;
// Per-tile cost of the heads task (a `big` task is 128).  It moves only 76 KB per tile but issues 24 N = 16 MMAs, each
// of which holds its issuing thread as long as a wide one (measured with a static item schedule: 2.08 / 1.76 / 1.65 /
// 1.65 / 1.63 ns per sample for the whole kernel at 50 / 80 / 110 / 140 / 178).
constexpr int kHeadsCost = 178;
// fp8 records (build_task_table8): 64 KB per tile for a `big` task (cost 128), 40 KB / 8 MMAs for the two encoding
// tasks, 38 KB / 12 narrow MMAs for the heads (swept on the GPU with 16 N = 128 MMAs per `big` tile,
// profiles/r02_fp8_records.md; those tiles now take 8 N = 256 MMAs)
constexpr int kXpartCost8 = 80;
constexpr int kHeadsCost8 = 94;
constexpr int kWMaxUnits = 6;
constexpr int kWQueue = 2;            // item ids in flight between the producer and the other roles
constexpr int kWBlocks = 4;           // TMEM accumulator blocks of 128 columns: flushed and handed back one at a time

// one ring slot: `bytes` from the forward (src 0) or dz (src 1) record at offset 0 and, optionally, `bytes2` from the
// dz record at slot offset 8192 (two small operands share a slot); bias_layer >= 0: column sums of this dZ unit
// are the bias gradient of that layer
struct WUnit { int src, off, bytes, bias_layer, bias_col0, off2, bytes2; };
// accumulator group: A = unit a (+ a_sub bytes), B = unit b (+ b_sub bytes)
struct WGroup { int a, b, col, N, layer, row_base, row_limit, col_base, mode, a_sub, b_sub, issuer; };
// last_grp[x][k]: the last group of issuer x that reads unit k (the one after which x releases the slot), -1 = none;
// last_in_blk[x][b]: the last group of issuer x in TMEM block b (its last tile's MMAs end the block's accumulation);
// a group covers the blocks blk_first(g) .. blk_last(g)
struct WTask {
  int n_units; WUnit u[kWMaxUnits]; int n_groups; WGroup g[kWMaxUnits]; int cost;
  int8_t last_grp[2][kWMaxUnits]; int8_t last_in_blk[2][kWBlocks];
};
// WGroup::mode, where the flush puts the accumulator:
enum : int {
  kFlushKernel = 0,   // dW[layer][(row_base+row), col_base+col] of a hidden layer
  kFlushHeads = 1,    // A = h7, B = the packed d_pre operand: column 3 = the sigma kernel's gradient, columns 0..2 =
                      // Y = h7^T d(rgb_pre) into the fp32 scratch
  kFlushDir = 4,      // A = PE(dir): columns 0..2 = Yd = PE(dir)^T d(rgb_pre) into the scratch (tc_finish_kernel uses Y, Yd)
};

struct WTaskTable { WTask t[kNumTasks]; };
// One accumulator group as its issuer runs it, built once per work item: units a / b, rel = release unit a (bit 0) /
// unit b (bit 1) after this group, cover / last = TMEM blocks the group writes / whose accumulation it ends for this
// issuer, slot-0 operand descriptors (with a_sub / b_sub), accumulator address, instruction descriptor.
struct IssueGroup { int a, b; uint32_t rel, cover, last; uint64_t da, db; uint32_t tcol, idesc; };
constexpr int kWMaxMine = 2;          // groups per issuer and task
__host__ __device__ inline int blk_first(const WGroup& g) { return g.col >> 7; }
__host__ __device__ inline int blk_last(const WGroup& g) { return (g.col + (g.N < 32 ? 32 : g.N) - 1) >> 7; }

// Fit the task table of the chain's fixed program to the model embedded in it (api.cu tc_chain_map).  Identity layers
// (w_off < 0) keep their tasks, so that the item layout does not depend on the model, but flush nothing: row_limit 0,
// no bias gradient.  A narrower model (U < 256) flushes only its own rows / columns, and the encoding rows of the
// concat layer start at row U of its kernel.
static void fit_tasks_to_model(WTaskTable& T, const TcParams& P) {
  for (int k = 0; k < kNumTasks; ++k) {
    WTask& t = T.t[k];
    for (int gi = 0; gi < t.n_groups; ++gi) {
      WGroup& g = t.g[gi];
      const int l = g.layer;
      if (g.mode == kFlushKernel && l >= 0 && l < 8) {
        if (l == 5 && g.row_base == 256) {            // encoding rows of the concat layer
          g.row_base = P.U;
          if (!P.x5) g.row_limit = 0;
        } else if (l > 0) {                           // hidden rows (layer 0's rows are encoding columns)
          g.row_limit = std::max(0, std::min(g.row_limit, P.U - g.row_base));
        }
        if (P.w_off[l] < 0) g.row_limit = 0;
      } else if (g.mode == kFlushHeads) {             // Y = h7^T d(rgb_pre) and the sigma kernel: rows of h7
        g.row_limit = std::max(0, std::min(g.row_limit, P.U - g.row_base));
      }
    }
    for (int u = 0; u < t.n_units; ++u)
      if (t.u[u].bias_layer >= 0 && P.b_off[t.u[u].bias_layer] < 0) t.u[u].bias_layer = -1;
  }
}

// Two MMA-issuing threads (tcgen05.mma holds its issuer for ~160 cycles per N = 128 MMA whose pipe time is 64):
// every accumulator group belongs to ONE issuer, so the fp32 accumulation order of each gradient element -- and
// with it every bit -- is that of a single issuer.  Default split: groups alternate (the heads task, the last one,
// sets its own).
static void finish_task_table(WTaskTable& T, int n) {
  for (int k = 0; k < n; ++k) {
    WTask& t = T.t[k];
    if (k != n - 1)
      for (int gi = 0; gi < t.n_groups; ++gi) t.g[gi].issuer = gi & 1;
    for (int x = 0; x < 2; ++x) {
      int mine = 0;
      for (int gi = 0; gi < t.n_groups; ++gi) mine += t.g[gi].issuer == x;
      if (mine > kWMaxMine) std::abort();   // the issuer keeps at most kWMaxMine groups in registers
    }
    for (int x = 0; x < 2; ++x) {
      for (int u = 0; u < kWMaxUnits; ++u) {
        t.last_grp[x][u] = -1;
        for (int gi = 0; gi < t.n_groups; ++gi)
          if (t.g[gi].issuer == x && (t.g[gi].a == u || t.g[gi].b == u)) t.last_grp[x][u] = (int8_t)gi;
      }
      for (int b = 0; b < kWBlocks; ++b) {
        t.last_in_blk[x][b] = -1;
        for (int gi = 0; gi < t.n_groups; ++gi)
          if (t.g[gi].issuer == x && blk_first(t.g[gi]) <= b && b <= blk_last(t.g[gi])) t.last_in_blk[x][b] = (int8_t)gi;
      }
    }
  }
}

static WTaskTable build_task_table(int dx, int dd) {
  WTaskTable T{};
  int n = 0;
  auto big = [&](int layer, int a_off, int b_off, int row_base) {   // A: two 128-feature halves, B: two 128-output halves
    WTask& t = T.t[n++];
    t.n_units = 4;
    t.u[0] = {0, a_off, kWUnitBytes, -1, 0}; t.u[1] = {1, b_off, kWUnitBytes, layer, 0};
    t.u[2] = {1, b_off + kWUnitBytes, kWUnitBytes, layer, 128}; t.u[3] = {0, a_off + kWUnitBytes, kWUnitBytes, -1, 0};
    t.n_groups = 4;
    t.g[0] = {0, 1, 0, 128, layer, row_base, 128, 0, kFlushKernel, 0, 0};
    t.g[1] = {0, 2, 128, 128, layer, row_base, 128, 128, kFlushKernel, 0, 0};
    t.g[2] = {3, 1, 256, 128, layer, row_base + 128, 128, 0, kFlushKernel, 0, 0};
    t.g[3] = {3, 2, 384, 128, layer, row_base + 128, 128, 128, kFlushKernel, 0, 0};
    t.cost = 128;
  };
  auto xpart = [&](int layer, int b_off, int row_base) {           // A: PE(xyz) (63 valid rows), B: two halves
    WTask& t = T.t[n++];
    t.n_units = 3;
    const int bl = (layer == 0) ? 0 : -1;   // layer 5's dZ column sums are taken by its h-part task
    // PE(xyz) is 64 features = 16 KB: only that much is fetched.  The MMA still reads a 128-feature unit; what the
    // rest of the ring slot holds (stale bytes) only reaches accumulator rows >= 64, which are never flushed.
    t.u[0] = {0, kRecXS, kXSBytes, -1, 0}; t.u[1] = {1, b_off, kWUnitBytes, bl, 0};
    t.u[2] = {1, b_off + kWUnitBytes, kWUnitBytes, bl, 128};
    t.n_groups = 2;
    t.g[0] = {0, 1, 0, 128, layer, row_base, dx, 0, kFlushKernel, 0, 0};
    t.g[1] = {0, 2, 128, 128, layer, row_base, dx, 128, kFlushKernel, 0, 0};
    t.cost = 76;    // costs = measured time per tile of a CTA working alone on the task (x 128 / the `big` tasks'):
                    // 3,700 / 6,300 / 8,400 cycles -- the kernel is bound by its CTAs' per-tile time, so equal item
                    // TIMES (not bytes) remove the tail
  };
  xpart(0, kDzZ0, 0);                                                        // layer 0
  for (int l = 1; l <= 7; ++l) big(l, kRecH0 + (l - 1) * kHSBytes, kDzZ0 + l * kHSBytes, 0);   // layers 1..7 (h part)
  xpart(5, kDzZ0 + 5 * kHSBytes, 256);                                       // layer 5, skip rows 256..318
  {  // Everything that hangs off h7 and d(rgb_features).  d(rgb_features) = dG = d(rgb_pre) Wc^T has rank 3, so every
     // gradient that contains it factors through three columns:  h7^T dG = (h7^T d(rgb_pre)) Wc^T,
     // PE(dir)^T dG = (PE(dir)^T d(rgb_pre)) Wc^T,  sum dG = (sum d(rgb_pre)) Wc^T.  The task therefore reads h7, PE(dir)
     // and the packed (d rgb_pre, d sigma_pre) operand only -- N = 16 MMAs -- and leaves Y = h7^T d(rgb_pre) [256 x 3]
     // (+ the sigma kernel's gradient, column 3 of the same accumulator) and Yd = PE(dir)^T d(rgb_pre) [27 x 3] in the
     // scratch, next to s3 = sum d(rgb_pre) from the dgrad prologue; tc_finish_kernel expands them into dW / db of
     // features, rgb_features and rgb.  Neither dG nor the rgb_features activations travel through HBM (64 KB per
     // tile less than round 1).
    WTask& t = T.t[n++];
    const int h7 = kRecH0 + 7 * kHSBytes;
    t.n_units = 3;
    t.u[0] = {0, h7, kWUnitBytes, -1, 0, 0, 0};                 // h7 features 0..127
    t.u[1] = {0, kRecDS, 8192, -1, 0, kDzP, 4096};              // PE(dir) (32 columns, 27 valid accumulator rows) and,
                                                                // at +8192, the packed (d rgb_pre, d sigma_pre) operand
    t.u[2] = {0, h7 + kWUnitBytes, kWUnitBytes, -1, 0, 0, 0};   // h7 features 128..255
    t.n_groups = 3;
    t.g[0] = {0, 1, 0, 16, 8, 0, 128, 0, kFlushHeads, 0, 8192};     // Y rows 0..127 (columns 0..2), sigma kernel (column 3)
    t.g[1] = {2, 1, 32, 16, 8, 128, 128, 0, kFlushHeads, 0, 8192};  // rows 128..255
    t.g[2] = {1, 1, 64, 16, -1, 0, dd, 0, kFlushDir, 0, 8192};      // Yd: A and B share the unit
    t.g[0].issuer = 0; t.g[1].issuer = 1; t.g[2].issuer = 0;
    t.cost = kHeadsCost;
  }
  finish_task_table(T, n);
  return T;
}

// fp8 records: a unit is a WHOLE 32 KB record (256 features x 128 samples); the accumulator groups address its halves
// through a_sub / b_sub.  64 KB per tile and `big` task instead of 128.
static WTaskTable build_task_table8(int dx, int dd) {
  WTaskTable T{};
  int n = 0;
  constexpr int kHalf = kH8Bytes / 2;
  auto big = [&](int layer, int a_off, int b_off, int row_base) {
    WTask& t = T.t[n++];
    t.n_units = 2;
    t.u[0] = {0, a_off, kH8Bytes, -1, 0, 0, 0}; t.u[1] = {1, b_off, kH8Bytes, layer, 0, 0, 0};
    // one N = 256 group per 128 input features: B is the whole record (its 16-column chunks are SBO apart, so both
    // halves of the outputs are one operand), and each issuer issues half as many MMAs as with 128 x 128 groups -- the
    // kernel is bound by MMA issue (profiles/r03_wgrad.md)
    t.n_groups = 2;
    t.g[0] = {0, 1, 0, 256, layer, row_base, 128, 0, kFlushKernel, 0, 0};
    t.g[1] = {0, 1, 256, 256, layer, row_base + 128, 128, 0, kFlushKernel, kHalf, 0};
    t.cost = 128;
  };
  auto xpart = [&](int layer, int b_off, int row_base) {
    WTask& t = T.t[n++];
    t.n_units = 2;
    const int bl = (layer == 0) ? 0 : -1;
    t.u[0] = {0, kRec8XS, 8192, -1, 0, 0, 0}; t.u[1] = {1, b_off, kH8Bytes, bl, 0, 0, 0};
    t.n_groups = 2;
    t.g[0] = {0, 1, 0, 128, layer, row_base, dx, 0, kFlushKernel, 0, 0};
    t.g[1] = {0, 1, 128, 128, layer, row_base, dx, 128, kFlushKernel, 0, kHalf};
    t.cost = kXpartCost8;
  };
  xpart(0, kDz8Z0, 0);
  for (int l = 1; l <= 7; ++l) big(l, kRec8H0 + (l - 1) * kH8Bytes, kDz8Z0 + l * kH8Bytes, 0);
  xpart(5, kDz8Z0 + 5 * kH8Bytes, 256);
  {
    WTask& t = T.t[n++];
    t.n_units = 2;
    t.u[0] = {0, kRec8H0 + 7 * kH8Bytes, kH8Bytes, -1, 0, 0, 0};   // h7
    t.u[1] = {0, kRec8DS, 4096, -1, 0, kDz8P, 2048};               // PE(dir) and, at +4096, the packed d_pre operand
    t.n_groups = 3;
    t.g[0] = {0, 1, 0, 16, 8, 0, 128, 0, kFlushHeads, 0, 4096};
    t.g[1] = {0, 1, 32, 16, 8, 128, 128, 0, kFlushHeads, kHalf, 4096};
    t.g[2] = {1, 1, 64, 16, -1, 0, dd, 0, kFlushDir, 0, 4096};
    t.g[0].issuer = 0; t.g[1].issuer = 1; t.g[2].issuer = 0;
    t.cost = kHeadsCost8;
  }
  finish_task_table(T, n);
  return T;
}

// ---- optional in-kernel counters (-DKNERF_TC_TIMING builds; knerf_debug_wgrad_timing reads them out) ----------------
// per CTA: 0 producer waits for a free slot (cycles) | 1, 2 issuer 0 / 1 waits for a loaded slot | 3, 4 issuer 0 / 1 waits
// for the previous item's flush | 5 flush warp 2: cycles from acc_done to its acc_free arrive | 6 flush warp 2 waits for
// acc_done | 7 items | 8 tiles | 9, 10 %globaltimer (ns) at the CTA's start / end | 11 CTA cycles start to end
// | 12, 13 issuer 0 / 1 cycles inside its MMA + commit sequences (its waits excluded) | 14 flush warp 2: cycles of the
// bias column sums | 15 dZ units column-summed | 16 flush warp 2 waits for a loaded slot | 17 flush warp 2 waits at the
// slot-release barrier of the four flush warps | 18, 19, 20 slot releases whose last arrival came from issuer 0 /
// issuer 1 / the flush warps | 21 releases where the flush warps arrived first | 22, 23 issuer 0 / 1 cycles from the end
// of one MMA + commit sequence to the start of the next group's waits (the loop's own instructions)
// (18-20: the flush warps' place is exact -- the pending count of the barrier state their arrive returns; between the
// two issuers the one that committed later counts as the later, since the MMAs of one SM complete in issue order)
#ifdef KNERF_TC_TIMING
constexpr int kWProf = 24;
static __device__ unsigned long long g_wg_prof[160][kWProf];
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define KN_WG_DECL() unsigned long long kn_wg[kWProf] = {}
#define KN_WG_WAIT(slot, bar, par) do { const long long kn_t0 = clock64(); mbar_wait(bar, par); \
                                        kn_wg[slot] += (unsigned long long)(clock64() - kn_t0); } while (0)
#define KN_WG_ADD(slot, v) kn_wg[slot] += (unsigned long long)(v)
#define KN_WG_CLOCK(var) const long long var = clock64()
#define KN_WG_FLUSH() for (int kn_i = 0; kn_i < kWProf; ++kn_i) if (kn_wg[kn_i]) atomicAdd(&g_wg_prof[blockIdx.x][kn_i], kn_wg[kn_i])
// mbarrier arrive that returns how many arrivals the phase still expected before this one (1: this one completed it)
__device__ __forceinline__ uint32_t mbar_arrive_pending(uint64_t* bar) {
  uint32_t n;
  asm volatile("{\n\t.reg .b64 st;\n\t"
               "mbarrier.arrive.shared::cta.b64 st, [%1];\n\t"
               "mbarrier.pending_count.b64 %0, st;\n\t}"
               : "=r"(n) : "r"(smem_u32(bar)) : "memory");
  return n;
}
#else
#define KN_WG_DECL()
#define KN_WG_WAIT(slot, bar, par) mbar_wait(bar, par)
#define KN_WG_ADD(slot, v)
#define KN_WG_CLOCK(var)
#define KN_WG_FLUSH()
#endif

struct WSmem {
  uint8_t slot[kWSlots][kWUnitBytes];
  uint64_t full[kWSlots], empty[kWSlots], acc_done[kWBlocks], acc_free[kWBlocks], q_full[kWQueue], q_empty[kWQueue];
  int q_item[kWQueue];
  uint32_t tmem_base;
  WUnit pu[kWMaxUnits];                // the producer's copy of the current task's units
#ifdef KNERF_TC_TIMING
  long long kn_commit_t[kWSlots][2];   // clock64 of each issuer's last release of the slot's current use
  int kn_flush_tag[kWSlots];           // (use << 1) | 1 if the flush warps' arrival completed the release
#endif
};

// Work items: (task, tiles [lo, hi)), claimed one at a time from a counter in the fp32 scratch (kXOffQueue) in the
// order of the list.  Boundaries depend only on n_tiles and the task costs, so every item's partial sums are the same
// bits from run to run; only the order of the cross-CTA red.global.add flushes varies, as it did with a static schedule.
constexpr int kWMaxItems = 1024;
struct WItemList { int2 range[kWMaxItems]; int8_t task[kWMaxItems]; };

// Guided sizes: an item takes 1/(kWGuide * 148) of the cost still unassigned, but no less than 1/kWMinShare of a CTA's
// share and no less than kWMinTiles `big` tiles (each item ends with a flush of up to 256 KB of partial sums), so items
// shrink towards the end of the list and the CTAs finish within about one small item of each other.  Items never span
// two tasks; the list is sorted longest first.
constexpr int kWGuide = 2;
constexpr int kWMinShare = 16;
constexpr int kWMinTiles = 4;
static int build_items(const WTaskTable& T, int64_t n_tiles, WItemList& L) {
  double total = 0.0;
  for (int k = 0; k < kNumTasks; ++k) total += (double)T.t[k].cost * (double)n_tiles;
  const double min_cost = std::max(total / kNumSMs / kWMinShare, 128.0 * kWMinTiles);
  struct It { double cost; int task; int64_t lo, hi; };
  std::vector<It> v;
  double left = total;
  for (int k = 0; k < kNumTasks; ++k) {
    const double c = T.t[k].cost;
    for (int64_t lo = 0; lo < n_tiles;) {
      const double want = std::max(min_cost, left / (kWGuide * kNumSMs));
      int64_t n = std::max<int64_t>(1, (int64_t)(want / c + 0.5));
      if (n_tiles - lo - n < (n + 1) / 2) n = n_tiles - lo;   // no runt at the end of a task
      v.push_back({c * (double)n, k, lo, lo + n});
      left -= c * (double)n;
      lo += n;
    }
  }
  std::stable_sort(v.begin(), v.end(), [](const It& a, const It& b) { return a.cost > b.cost; });
  if ((int64_t)v.size() > kWMaxItems) return -1;
  for (size_t i = 0; i < v.size(); ++i) {
    L.range[i] = make_int2((int)v[i].lo, (int)v[i].hi);
    L.task[i] = (int8_t)v[i].task;
  }
  return (int)v.size();
}

// Roles: warp 0 lane 0 claims items and loads their operand units into the ring; warps 1 and 6 (lane 0) issue the MMAs
// of their accumulator groups; warps 2-5 take the bias gradients while an item runs and flush its accumulators after it.
// The item ids reach the other roles through a kWQueue-deep shared-memory queue (the producer runs ahead into the next
// item while the current one is being computed).  TMEM block b (128 columns) of the next item is written only after the
// flush warps have drained block b of the previous one (acc_free[b]); they drain block 0 first.
template <bool REC8>
__global__ void __launch_bounds__(kWThreads, 1)
tc_wgrad_kernel(const uint8_t* __restrict__ rec, const uint8_t* __restrict__ dz, float* __restrict__ grads,
                float* __restrict__ xbuf, TcParams P, const __grid_constant__ WTaskTable T,
                const __grid_constant__ WItemList L, int n_items) {
  constexpr int kRB = REC8 ? kRec8Bytes : kRecBytes, kDB = REC8 ? kDz8Bytes : kDzBytes;
  constexpr int kSub2 = REC8 ? 4096 : 8192;   // slot offset of a unit's second part (the packed d_pre operand)
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  WSmem& sm = *reinterpret_cast<WSmem*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  KN_WG_DECL();
  KN_WG_CLOCK(kn_start);
#ifdef KNERF_TC_TIMING
  if (tid == 0) g_wg_prof[blockIdx.x][9] = globaltimer_ns();
#endif
  if (tid == 0) {
    // a slot is free again when the MMAs that read it have completed AND the flush warps are done with it
    // (one release per issuer + one from the flush warps)
    for (int i = 0; i < kWSlots; ++i) { mbar_init(&sm.full[i], 1); mbar_init(&sm.empty[i], 3); }
    for (int b = 0; b < kWBlocks; ++b) { mbar_init(&sm.acc_done[b], 2); mbar_init(&sm.acc_free[b], 128); }
    // a queue entry is read by the two issuers and the four flush warps
    for (int i = 0; i < kWQueue; ++i) { mbar_init(&sm.q_full[i], 1); mbar_init(&sm.q_empty[i], 6); }
#ifdef KNERF_TC_TIMING
    for (int i = 0; i < kWSlots; ++i) sm.kn_flush_tag[i] = -2;
#endif
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<512>(&sm.tmem_base);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = sm.tmem_base;
  // the j-th item of this CTA (-1: none left)
  auto take_item = [&](int j) -> int {
    mbar_wait(&sm.q_full[j % kWQueue], (j / kWQueue) & 1);
    return *reinterpret_cast<volatile int*>(&sm.q_item[j % kWQueue]);
  };

  if (warp == 0) {
    if (lane == 0) {
      unsigned int* counter = reinterpret_cast<unsigned int*>(xbuf + kXOffQueue);
      uint32_t it = 0;
      for (int j = 0;; ++j) {
        const int claimed = (int)atomicAdd(counter, 1u);
        const int item = claimed < n_items ? claimed : -1;
        mbar_wait(&sm.q_empty[j % kWQueue], ((j / kWQueue) & 1) ^ 1);
        sm.q_item[j % kWQueue] = item;
        mbar_arrive(&sm.q_full[j % kWQueue]);
        if (item < 0) break;
        const WTask& t = T.t[L.task[item]];
        const int n_units = t.n_units;
        for (int k = 0; k < n_units; ++k) sm.pu[k] = t.u[k];   // (indexed constant-bank reads are slow: once per item)
        for (int64_t tile = L.range[item].x; tile < L.range[item].y; ++tile) {
          for (int k = 0; k < n_units; ++k, ++it) {
            const WUnit u = sm.pu[k];
            const uint32_t slot = it % kWSlots, ph = (it / kWSlots) & 1;
            const uint8_t* src = (u.src == 0 ? rec + tile * kRB : dz + tile * kDB) + u.off;
            KN_WG_WAIT(0, &sm.empty[slot], ph ^ 1);
#ifdef KNERF_TC_TIMING
            if (it >= (uint32_t)kWSlots) {   // who released use it / kWSlots - 1 of this slot last
              const int tag = *reinterpret_cast<volatile int*>(&sm.kn_flush_tag[slot]);
              const volatile long long* ct = sm.kn_commit_t[slot];
              // a tag not yet written for this use: the flush warps' arrival was the one that just completed it
              if ((tag >> 1) != (int)(it / kWSlots - 1) || (tag & 1)) KN_WG_ADD(20, 1);
              else KN_WG_ADD(ct[0] > ct[1] ? 18 : 19, 1);
            }
#endif
            mbar_arrive_expect_tx(&sm.full[slot], u.bytes + u.bytes2);
            tma_load_1d(sm.slot[slot], src, u.bytes, &sm.full[slot]);
            if (u.bytes2) tma_load_1d(sm.slot[slot] + kSub2, dz + tile * kDB + u.off2, u.bytes2, &sm.full[slot]);
          }
        }
      }
    }
  } else if (warp == 1 || warp == 6) {
    if (lane == 0) {
      const int me = (warp == 1) ? 0 : 1;
      const uint32_t slot0 = smem_u32(sm.slot[0]);
      uint32_t it = 0;
#ifdef KNERF_TC_TIMING
      long long kn_mark = clock64();
#endif
      for (int j = 0;; ++j) {
        const int item = take_item(j);
        mbar_arrive(&sm.q_empty[j % kWQueue]);
        if (item < 0) break;
        const WTask& t = T.t[L.task[item]];
        const int64_t lo = L.range[item].x, hi = L.range[item].y;
        // This issuer's part of the task, read from the table once per item: the table lives in the constant bank,
        // and the indexed reads of it in the tile loop held the issuer ~1,150 cycles per tile
        // (profiles/r04_wgrad_limiter.md).
        IssueGroup mine[kWMaxMine];
        int n_mine = 0;
        uint32_t skip = 0;   // units this issuer never reads
        for (int k = 0; k < t.n_units; ++k)
          if (t.last_grp[me][k] < 0) skip |= 1u << k;
        for (int gi = 0; gi < t.n_groups; ++gi) {
          const WGroup& g = t.g[gi];
          if (g.issuer != me) continue;
          IssueGroup m;
          m.a = g.a; m.b = g.b;
          m.rel = (t.last_grp[me][g.a] == gi ? 1u : 0u) | (g.b != g.a && t.last_grp[me][g.b] == gi ? 2u : 0u);
          m.cover = 0u; m.last = 0u;
          for (int b = blk_first(g); b <= blk_last(g); ++b) {
            m.cover |= 1u << b;
            if (t.last_in_blk[me][b] == gi) m.last |= 1u << b;   // this group ends this issuer's part of block b
          }
          m.da = umma_smem_desc(slot0 + g.a_sub, 128, kChunkA);
          m.db = umma_smem_desc(slot0 + g.b_sub, 128, kChunkA);
          m.tcol = tmem + g.col;
          m.idesc = REC8 ? umma_idesc_f8(128, g.N, kE4M3, kE5M2, 1, 1) : umma_idesc_bf16(128, g.N, 1, 1);
          if (n_mine == 0) mine[0] = m; else mine[1] = m;   // constant indices keep `mine` in registers
          ++n_mine;
        }
        const int n_units = t.n_units;
        // Block b of this item may be written once the flush warps have drained it for the previous item.  Every item
        // waits for all blocks (those it does not write at its end, before its acc_done arrival), so that neither
        // barrier of a block can get a phase ahead of its reader.
        uint32_t freed = (j == 0) ? 0xFu : 0u, done = 0u;
        auto wait_free = [&](int b) {
          if (!((freed >> b) & 1u)) {
            KN_WG_WAIT(3 + me, &sm.acc_free[b], (j - 1) & 1);
            tc_fence_after();
            freed |= 1u << b;
          }
        };
        auto issue = [&](const IssueGroup& m, int64_t tile) {
#ifdef KNERF_TC_TIMING
          KN_WG_ADD(22 + me, clock64() - kn_mark);
#endif
          if (tile == lo)
            for (int b = 0; b < kWBlocks; ++b)
              if ((m.cover >> b) & 1u) wait_free(b);
          const uint32_t ia = it + m.a, ib = it + m.b;
          const uint32_t sa = ia % kWSlots, sb = ib % kWSlots;
          KN_WG_WAIT(1 + me, &sm.full[sa], (ia / kWSlots) & 1);
          KN_WG_WAIT(1 + me, &sm.full[sb], (ib / kWSlots) & 1);
          KN_WG_CLOCK(kn_issue);
          tc_fence_after();
          // the descriptors' start-address field is addr >> 4 (< 2^14 for any shared-memory address): slot and k
          // offsets add to the precomputed slot-0 descriptors
          const uint64_t da = m.da + (uint64_t)(sa * (kWUnitBytes >> 4)), db = m.db + (uint64_t)(sb * (kWUnitBytes >> 4));
          if (REC8) {   // e4m3 activations x e5m2 gradients, 32 samples per MMA (512 B further along every chunk)
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_f8(m.tcol, da + k * 32, db + k * 32, m.idesc, (tile > lo || k > 0) ? 1u : 0u);
          } else {
#pragma unroll
            for (int k = 0; k < 8; ++k)   // K = 128 samples per tile, 16 per MMA; MN-major: LBO = 128 B, SBO = 2 KB
              umma_bf16(m.tcol, da + k * 16, db + k * 16, m.idesc, (tile > lo || k > 0) ? 1u : 0u);
          }
#ifdef KNERF_TC_TIMING
          if (m.rel & 1u) sm.kn_commit_t[sa][me] = clock64();
          if (m.rel & 2u) sm.kn_commit_t[sb][me] = clock64();
#endif
          if (m.rel & 1u) umma_commit(&sm.empty[sa]);
          if (m.rel & 2u) umma_commit(&sm.empty[sb]);
          if (tile + 1 == hi && m.last) {
            for (int b = 0; b < kWBlocks; ++b)
              if ((m.last >> b) & 1u) umma_commit(&sm.acc_done[b]);
            done |= m.last;
          }
          KN_WG_ADD(12 + me, clock64() - kn_issue);
#ifdef KNERF_TC_TIMING
          kn_mark = clock64();
#endif
        };
        for (int64_t tile = lo; tile < hi; ++tile, it += n_units) {
          if (n_mine > 0) issue(mine[0], tile);
          if (n_mine > 1) issue(mine[1], tile);
          // units this issuer never reads: release them too (after their load has landed, so that the arrival
          // counts for this use of the slot and not for the previous one)
          for (uint32_t sk = skip; sk != 0u; sk &= sk - 1u) {
            const uint32_t iu = it + (uint32_t)(__ffs(sk) - 1);
            mbar_wait(&sm.full[iu % kWSlots], (iu / kWSlots) & 1);
#ifdef KNERF_TC_TIMING
            sm.kn_commit_t[iu % kWSlots][me] = clock64();
#endif
            mbar_arrive(&sm.empty[iu % kWSlots]);
          }
        }
        for (int b = 0; b < kWBlocks; ++b) {
          if ((done >> b) & 1u) continue;
          wait_free(b);
          umma_commit(&sm.acc_done[b]);
        }
      }
    }
  } else {
    // flush warps: TMEM lane quadrant = warp & 3
    const int q = warp & 3, row = q * 32 + lane;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    const int ftid = tid - 64, fc = ftid >> 3, fsub = ftid & 7;
    const float inv_scale = REC8 ? dz8_scale(__ldg(reinterpret_cast<const uint32_t*>(xbuf) + kXOffAmax), true) : 1.f;
    uint32_t uit = 0;
    for (int j = 0;; ++j) {
      const int item = take_item(j);
      __syncwarp();
      if (lane == 0) mbar_arrive(&sm.q_empty[j % kWQueue]);
      if (item < 0) break;
      const WTask& t = T.t[L.task[item]];
      const int64_t lo = L.range[item].x, hi = L.range[item].y;
      // While the tensor core works through the item, these warps take the bias gradients: column sums (over
      // samples) of every dZ unit passing through shared memory.  Thread (fc, fsub) owns 8 columns of chunk fc
      // and every 8th sample; partial sums stay in registers for the whole item.
      // (fp8 records: a task has ONE dZ unit of 16 chunks x 16 columns; bacc[0] / bacc[1] = columns 0..7 / 8..15 of chunk fc)
      float bacc[2][8];
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int e = 0; e < 8; ++e) bacc[u][e] = 0.f;
      for (int64_t tile = lo; tile < hi; ++tile) {
        int nb = 0;
        for (int k = 0; k < t.n_units; ++k, ++uit) {
          const uint32_t slot = uit % kWSlots;
          KN_WG_WAIT(16, &sm.full[slot], (uit / kWSlots) & 1);
          KN_WG_CLOCK(kn_bias);
          if (t.u[k].bias_layer >= 0) {
            KN_WG_ADD(15, 1);
            const uint8_t* base = sm.slot[slot] + fc * kChunkA + fsub * 16;
            if (REC8) {
#pragma unroll 4
              for (int i = 0; i < 16; ++i) {
                const uint4 v = *reinterpret_cast<const uint4*>(base + i * 128);
                const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) add_e5m2x4(bacc[jj >> 1] + (jj & 1) * 4, wv[jj]);
              }
            } else {
              float* a = bacc[nb & 1];
#pragma unroll 4
              for (int i = 0; i < 16; ++i) {
                const uint4 v = *reinterpret_cast<const uint4*>(base + i * 128);
                a[0] += bf16_lo(v.x); a[1] += bf16_hi(v.x); a[2] += bf16_lo(v.y); a[3] += bf16_hi(v.y);
                a[4] += bf16_lo(v.z); a[5] += bf16_hi(v.z); a[6] += bf16_lo(v.w); a[7] += bf16_hi(v.w);
              }
            }
            ++nb;
          }
#ifdef KNERF_TC_TIMING
          const long long kn_sum_end = clock64();
          KN_WG_ADD(14, kn_sum_end - kn_bias);
          named_bar_sync(2, 128);
          KN_WG_ADD(17, clock64() - kn_sum_end);
          if (ftid == 0) {
            const uint32_t pending = mbar_arrive_pending(&sm.empty[slot]);
            sm.kn_flush_tag[slot] = (int)((uit / kWSlots) << 1) | (pending == 1 ? 1 : 0);
            if (pending == 3) KN_WG_ADD(21, 1);
          }
#else
          named_bar_sync(2, 128);               // all 128 readers are done with the slot
          if (ftid == 0) mbar_arrive(&sm.empty[slot]);
#endif
        }
      }
      {
        int nb = 0;
        for (int k = 0; k < t.n_units; ++k) {
          if (t.u[k].bias_layer < 0) continue;
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            if (!REC8 && u != (nb & 1)) continue;
            float* a = bacc[u];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              a[e] += __shfl_xor_sync(0xffffffffu, a[e], 1);
              a[e] += __shfl_xor_sync(0xffffffffu, a[e], 2);
              a[e] += __shfl_xor_sync(0xffffffffu, a[e], 4);
            }
            if (fsub == 0) {
              const int c0 = t.u[k].bias_col0 + (REC8 ? fc * 16 + u * 8 : fc * 8);
              float* dst = grads + P.b_off[t.u[k].bias_layer] + c0;
#pragma unroll
              for (int e = 0; e < 8; ++e)
                if (c0 + e < P.U) atomicAdd(dst + e, a[e] * inv_scale);
            }
          }
          ++nb;
        }
      }
      KN_WG_ADD(7, 1);
      KN_WG_ADD(8, hi - lo);
      for (int b = 0; b < kWBlocks; ++b) {
        KN_WG_WAIT(6, &sm.acc_done[b], j & 1);
        KN_WG_CLOCK(kn_flush);
        tc_fence_after();
        for (int gi = 0; gi < t.n_groups; ++gi) {
          const WGroup& g = t.g[gi];
          const int ncol = g.N < 32 ? 32 : g.N;
          for (int c0 = 0; c0 < ncol; c0 += 32) {
            if (((g.col + c0) >> 7) != b) continue;
            float v[32];
            tmem_ld32(tmem + lane_base + g.col + c0, v);   // warp-collective: outside the row guard
            if (REC8) {
#pragma unroll
              for (int i = 0; i < 32; ++i) v[i] *= inv_scale;
            }
            if (row < g.row_limit) {
              if (g.mode == kFlushKernel) {   // kernel [fan_in, U] of a hidden layer: columns >= U belong to the padding
                float* dst = grads + P.w_off[g.layer] + (int64_t)(g.row_base + row) * P.U + g.col_base + c0;
                const int nv = P.U - (g.col_base + c0);
                if (nv >= 32 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
#pragma unroll
                  for (int i = 0; i < 32; i += 4) red_add_v4(dst + i, v[i], v[i + 1], v[i + 2], v[i + 3]);
                } else {   // a narrower model's last columns, or a row that does not start 16-byte aligned
#pragma unroll
                  for (int i = 0; i < 32; ++i)
                    if (i < nv) atomicAdd(dst + i, v[i]);
                }
              } else if (g.mode == kFlushHeads) {
                atomicAdd(grads + P.w_off[8] + g.row_base + row, v[3]);
                float* dst = xbuf + kXOffY + (g.row_base + row) * 4;
                atomicAdd(dst, v[0]); atomicAdd(dst + 1, v[1]); atomicAdd(dst + 2, v[2]);
              } else {
                float* dst = xbuf + kXOffYd + row * 4;
                atomicAdd(dst, v[0]); atomicAdd(dst + 1, v[1]); atomicAdd(dst + 2, v[2]);
              }
            }
          }
        }
        tc_fence_before();
        mbar_arrive(&sm.acc_free[b]);
        KN_WG_ADD(5, clock64() - kn_flush);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<512>(tmem);
#ifdef KNERF_TC_TIMING
  if (tid == 0) {
    KN_WG_ADD(11, clock64() - kn_start);
    g_wg_prof[blockIdx.x][10] = globaltimer_ns();
  }
  if (tid == 0 || tid == 32 || tid == 64 || tid == 192) KN_WG_FLUSH();
#endif
}

// =============================================================================================================
// heads: features / rgb_features / rgb gradients from the rank-3 factors
// =============================================================================================================
// With Y = h7^T d(rgb_pre) [256 x 3], Yd = PE(dir)^T d(rgb_pre) [27 x 3], s3 = sum d(rgb_pre) [3] of THIS call (scratch,
// 4 floats per row) and the weights W_f [256,256], b_f, W_g [283,128], W_c [128,3], W' = W_f W_g[:256], b' (fold):
//   X = h7^T dG = Y W_c^T,  sum dG = s3 W_c^T   (never formed: T[j][c] = sum_n W_g[j][n] W_c[n][c],
//                                                U[j][c] = sum_i W_f[i][j] Y[i][c] + b_f[j] s3[c])
//   dW_f[i][j]        += sum_c Y[i][c] T[j][c]                    db_f[j]  += sum_c s3[c] T[j][c]
//   dW_g[j][n]        += sum_c U[j][c] W_c[n][c]      (j < 256)   db_g[n]  += sum_c s3[c] W_c[n][c]
//   dW_g[256 + i][n]  += sum_c Yd[i][c] W_c[n][c]     (i < 27)
//   dW_c[k][c]        += sum_j W'[j][k] Y[j][c] + sum_i W_g[256+i][k] Yd[i][c] + b'[k] s3[c]
// tc_finish_prep_kernel forms T and U (256 x 3 each), tc_finish_kernel one output element per thread.
constexpr int kFinF = 256 * 256, kFinG = 256 * 128, kFinBf = 256, kFinGd = 27 * 128, kFinBg = 128, kFinC = 128 * 3;   // (kFinGd: rows >= dd idle)
constexpr int kFinTotal = kFinF + kFinG + kFinBf + kFinGd + kFinBg + kFinC;

// the two U x 3 factors every output of tc_finish_kernel needs (one thread each; 0.3 M MAC)
// (U = dense_units <= 256, H = U / 2: the kernels are [U, U], [U + dd, H], [H, 3] in the flat buffer; the scratch and the
//  fold keep their 256 / 128 strides)
__global__ void __launch_bounds__(256) tc_finish_prep_kernel(const float* __restrict__ params, TcParams P,
                                                             float* __restrict__ xbuf) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;   // < 2 * 256 * 3
  const int which = idx / 768, e = idx - which * 768, j = e / 3, c = e - j * 3;
  const int U = P.U, H = P.U / 2;
  if (which > 1) return;
  const float* Wc = params + P.w_off[11];
  float acc = 0.f;
  if (which == 0) {
    if (j < U) {
      const float* w = params + P.w_off[10] + (int64_t)j * H;
      for (int n = 0; n < H; ++n) acc = fmaf(w[n], Wc[n * 3 + c], acc);
    }
    xbuf[kXOffT + j * 4 + c] = acc;
  } else {
    if (j < U) {
      const float* Wf = params + P.w_off[9];
      const float* Y = xbuf + kXOffY;
      acc = params[P.b_off[9] + j] * xbuf[kXOffS + c];
      for (int i = 0; i < U; ++i) acc = fmaf(Wf[(int64_t)i * U + j], Y[i * 4 + c], acc);
    }
    xbuf[kXOffU + j * 4 + c] = acc;
  }
}

__global__ void __launch_bounds__(256) tc_finish_kernel(const float* __restrict__ params, TcParams P,
                                                        const float* __restrict__ xbuf, float* __restrict__ grads,
                                                        const float* __restrict__ fold) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int U = P.U, H = P.U / 2;
  const float* Wg = params + P.w_off[10];   // rgb_features  [U + dd, H]
  const float* Wc = params + P.w_off[11];   // rgb           [H, 3]
  const float* Y = xbuf + kXOffY;
  const float* Yd = xbuf + kXOffYd;
  const float* T = xbuf + kXOffT;
  const float* Uf = xbuf + kXOffU;
  const float s3[3] = {xbuf[kXOffS], xbuf[kXOffS + 1], xbuf[kXOffS + 2]};
  if (idx < kFinF) {
    const int i = idx >> 8, j = idx & 255;
    if (i < U && j < U)
      grads[P.w_off[9] + (int64_t)i * U + j] += Y[i * 4] * T[j * 4] + Y[i * 4 + 1] * T[j * 4 + 1] + Y[i * 4 + 2] * T[j * 4 + 2];
    return;
  }
  idx -= kFinF;
  if (idx < kFinG) {
    const int j = idx >> 7, n = idx & 127;
    if (j < U && n < H)
      grads[P.w_off[10] + (int64_t)j * H + n] += Uf[j * 4] * Wc[n * 3] + Uf[j * 4 + 1] * Wc[n * 3 + 1] + Uf[j * 4 + 2] * Wc[n * 3 + 2];
    return;
  }
  idx -= kFinG;
  if (idx < kFinBf) {
    if (idx < U) grads[P.b_off[9] + idx] += s3[0] * T[idx * 4] + s3[1] * T[idx * 4 + 1] + s3[2] * T[idx * 4 + 2];
    return;
  }
  idx -= kFinBf;
  if (idx < kFinGd) {
    const int i = idx >> 7, n = idx & 127;
    if (i < P.dd && n < H)
      grads[P.w_off[10] + (int64_t)(U + i) * H + n] += Yd[i * 4] * Wc[n * 3] + Yd[i * 4 + 1] * Wc[n * 3 + 1] + Yd[i * 4 + 2] * Wc[n * 3 + 2];
    return;
  }
  idx -= kFinGd;
  if (idx < kFinBg) {
    if (idx < H) grads[P.b_off[10] + idx] += s3[0] * Wc[idx * 3] + s3[1] * Wc[idx * 3 + 1] + s3[2] * Wc[idx * 3 + 2];
    return;
  }
  idx -= kFinBg;
  if (idx < kFinC) {
    const int k = idx / 3, c = idx - k * 3;
    if (k >= H) return;
    float acc = fold[256 * 128 + k] * s3[c];
    for (int j = 0; j < U; ++j) acc = fmaf(fold[j * 128 + k], Y[j * 4 + c], acc);
    for (int i = 0; i < P.dd; ++i) acc = fmaf(Wg[(int64_t)(U + i) * H + k], Yd[i * 4 + c], acc);
    grads[P.w_off[11] + idx] += acc;
  }
}

}  // namespace

// diagnostic (-DKNERF_TC_TIMING builds only): copy and clear the weight-gradient kernel's per-CTA counters
int tc_debug_wgrad_timing(unsigned long long* host_out, int n) { return KN_PROF_READ(g_wg_prof, host_out, n); }

// diagnostic (-DKNERF_TC_TIMING builds only): copy and clear the dgrad kernel's per-CTA cycle counters (the slots of
// tc_roles.cuh; this translation unit has its own g_tc_prof, so the forward's counters do not mix in)
int tc_debug_dgrad_timing(unsigned long long* host_out, int n) { return KN_PROF_READ(g_tc_prof, host_out, n); }

// parts: which of the backward kernels to launch (bit 0 dgrad, bit 1 wgrad + finish; KNERF_BWD_*_ONLY)
int tc_backward(const Model& m, const float* params, const void* packed, const float* d_pre, int64_t R, int S,
                float* grads, char* ws, int64_t ws_bytes, int parts, bool rec8, cudaStream_t st) {
  if (!is_flagship(m)) return fail(KNERF_ERR_UNSUPPORTED, "KNERF_BF16 implements models of dense_units <= 256 (even), up to 8 layers, at most one skip concat (not into the heads), L_xyz <= 10, L_dir <= 4");
  KN_CHECK_ARG(packed != nullptr, "KNERF_BF16 needs packed weights (knerf_pack_weights)");
  const int64_t M = R * S;
  if (ws_bytes < tc_workspace_bytes(m, M, true, rec8))
    return fail(KNERF_ERR_WORKSPACE, "tc_backward: workspace %lld < %lld bytes", (long long)ws_bytes,
                (long long)tc_workspace_bytes(m, M, true, rec8));
  KN_CHECK_ARG((reinterpret_cast<uintptr_t>(d_pre) & 15) == 0, "tc_backward: d_pre must be 16-byte aligned");
  const int64_t n_tiles = cdiv(M, kTileM);
  float* xbuf = (float*)ws;                                // X = h7^T dG and sum(dG) of this call
  uint8_t* rec = (uint8_t*)ws + kXBytes;
  uint8_t* dz = rec + n_tiles * (int64_t)(rec8 ? kRec8Bytes : kRecBytes);
  const TcParams P = tc_make_params(m);
  // the fp32 scratch (rank-3 factors, sum d(rgb_pre), max|d_pre|) starts from zero in every call -- except that a
  // weight-gradient-only call (KNERF_BWD_WGRAD_ONLY) keeps what the dgrad-only call before it left there: sum d(rgb_pre)
  // and (fp8 records) the scale of the gradient records
  KN_CUDA(cudaMemsetAsync(xbuf, 0, (parts == 2 ? kXOffS : kXFloats) * sizeof(float), st));

  if (parts & 1) {
    const float4* dp = (const float4*)d_pre;
    if (rec8) {
      dpre_amax_kernel<<<kNumSMs * 4, 256, 0, st>>>(dp, M, reinterpret_cast<uint32_t*>(xbuf) + kXOffAmax);
      KN_LAUNCH_CHECK();
    }
    KN_TRY(launch_chain(rec8 ? &tc_mlp_dgrad_kernel<true> : &tc_mlp_dgrad_kernel<false>, n_tiles, st,
                        (const uint8_t*)packed, dp, M, (const uint8_t*)rec, dz, grads, P, xbuf));
  }
  if (parts & 2) {
    // the task table (~3 KB) and the item list (~9 KB) are passed by value as __grid_constant__ parameters
    WTaskTable h_table = rec8 ? build_task_table8(m.dx, m.dd) : build_task_table(m.dx, m.dd);
    fit_tasks_to_model(h_table, P);
    KN_CHECK_ARG(n_tiles < (int64_t)1 << 30, "tc_backward: %lld rows are too many for one call", (long long)M);
    WItemList h_items;
    const int n_items = build_items(h_table, n_tiles, h_items);
    if (n_items < 0) return fail(KNERF_ERR_UNSUPPORTED, "tc_backward: more than %d weight-gradient items", kWMaxItems);
    const size_t smem = sizeof(WSmem);
    auto wgrad = rec8 ? &tc_wgrad_kernel<true> : &tc_wgrad_kernel<false>;
    KN_CUDA(cudaFuncSetAttribute(wgrad, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    wgrad<<<kNumSMs, kWThreads, smem, st>>>(rec, dz, grads, xbuf, P, h_table, h_items, n_items);
    KN_LAUNCH_CHECK();
    tc_finish_prep_kernel<<<6, 256, 0, st>>>(params, P, xbuf);
    KN_LAUNCH_CHECK();
    tc_finish_kernel<<<(kFinTotal + 255) / 256, 256, 0, st>>>(
        params, P, xbuf, grads, reinterpret_cast<const float*>((const uint8_t*)packed + kFoldOff));
    KN_LAUNCH_CHECK();
  }
  return KNERF_OK;
}

}  // namespace knerf
