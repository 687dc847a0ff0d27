// Shapes, step tables and HBM layouts shared by the tcgen05 forward (mlp_tc.cu) and backward
// (mlp_tc_bwd.cu) kernels.  ONE program -- eight 256-wide layers, the encoding concatenated in front of layer 5 -- into
// which the models csrc/api.cu tc_chain_map accepts are embedded (fewer layers: identity layers; fewer frequencies: zero rows).
#pragma once

#include <stdint.h>

namespace knerf {
namespace tcl {

constexpr int kTileM = 128;                        // samples per tile (UMMA M per CTA)
constexpr int kU = 256;
constexpr int kKStage = 32;                        // granularity of the K tables below (nk_h / nk_x count 32-wide blocks)
constexpr int kHSBytes = kTileM * kU * 2;          // 64 KB: one [128 x 256] bf16 operand, chunk-major
constexpr int kXSBytes = kTileM * 64 * 2;          // 16 KB
constexpr int kChunkA = kTileM * 16;               // bytes between 8-element chunks of a 128-row operand (2048)
constexpr int kThreads = 384;                      // warps: 0 TMA producer, 1 MMA issuer (even ring items) / relay,
                                                   // 2-9 compute, 10 record store (training kernels), 11 MMA issuer of
                                                   // the odd ring items (leader CTA).  12 warps: a 13th would cap ptxas
                                                   // at 128 registers and spill (no L1 here: a spill is an L2 trip)
constexpr int kComputeThreads = 256;

// ---- forward steps ---------------------------------------------------------------------------------------
// mlp.py:42-46 applies NO activation between `features` and `rgb_features`, so
//   G = [h7 W_f + b_f, dir] W_g + b_g = h7 (W_f W_g[:256]) + dir W_g[256:] + (b_f W_g[:256] + b_g)
// is ONE step from h7 (the product W' = W_f W_g[:256] is formed in fp32 when the weights are packed).  Saves the
// 256 x 256 `features` GEMM (11 % of the MACs) and its 64 KB/tile activation record.  The rgb head after it is linear
// too (mlp.py:47-48: sigmoid(G W_c + b_c)), so the last step goes from h7 straight to the head pre-activations:
//   rgb_pre = h7 W''' + PE(dir) D + b'''      W''' = W' W_c [256 x 3],  D = W_g[256:] W_c [27 x 3],  b''' = b' W_c + b_c
// (formed in fp32 at packing, fold_kernel), and sigma_pre = h7 w_s + b_s rides along as output column 3.  Columns 4..7
// repeat the four with the bf16 residual of each weight (mlp_tc.cu fold_weight): N = 16, the epilogue adds column
// pairs and applies the sigmoids and the ReLU.
// The backward pass never needs the `features` activations either: with X = h7^T dG (one weight-gradient GEMM)
//   dW_f = X W_g[:256]^T,   dW_g[:256] = W_f^T X + b_f (x) sum(dG),   db_f = sum(dG) W_g[:256]^T
// (tc_finish_kernel, once per backward call), and the dgrad chain goes from dG to d(h7) through W'^T directly.
// Reported FLOP counts always use the unfolded 593,408 MAC per sample (SURVEY §8d).
// step:        0    1..4   5      6,7   8
// layer:       L0   L1-4   L5     L6,7  [rgb o rgb_features o features | sigma]
struct FwdProg {
  static constexpr int kSteps = 9;
  static constexpr int kNLast = 16;                  // (rgb_pre[3], sigma_pre) x (bf16 part, residual), 8 zero columns
  __host__ __device__ static constexpr int layer(int s) { return s; }   // (s < 8; the last step is packed specially)
  __host__ __device__ static constexpr int nk_h(int s) { return s == 0 ? 0 : 8; }   // 32-wide K blocks fed by hs
  __host__ __device__ static constexpr int nk_x(int s) { return (s == 0 || s == 5) ? 2 : (s == 8 ? 1 : 0); }
  __host__ __device__ static constexpr int N(int s) { return s == 8 ? kNLast : 256; }
  // Bias folded into the GEMM: every step ends with ONE extra K=16 MMA whose A operand is two chunks of the
  // encoding buffer that contain a constant-1 column (PE(xyz) pad column 63 for steps 0..5, PE(dir) pad column
  // 31 afterwards) and whose B operand [2 chunks][N][8] is zero except k = 15 <- bias[n].  The real weight rows
  // of those pad columns are zero, so the 1.0 never leaks into the ordinary stages.  Costs 1/16 more MMA time,
  // removes every bias load and add from the epilogue (which is the critical path).
  static constexpr bool kHasBias = true;
  __host__ __device__ static constexpr int bias_a_chunk(int s) { return s <= 5 ? 6 : 2; }
};

// ---- backward (dgrad) steps --------------------------------------------------------------------------------
// step b:      0                                                          1 .. 7
// computes:    dZ7 = (d(rgb_pre) W'''^T + dsigma Ws^T) * [h7>0]           dZ_{7-b} = (dZ_{8-b} W_{8-b}^T) * [h_{7-b}>0]
// weights:     [W''' | Ws | 0] (K = 32: d rgb_pre[3], d sigma_pre, zeros)  layer 7 .. layer 1   (rows < 256 of the Keras kernel)
struct BwdProg {
  static constexpr int kSteps = 8;
  __host__ __device__ static constexpr int layer(int b) { return 8 - b; }            // (b >= 1)
  __host__ __device__ static constexpr int nk_h(int b) { return b == 0 ? 1 : 8; }
  __host__ __device__ static constexpr int nk_x(int) { return 0; }
  __host__ __device__ static constexpr int N(int) { return 256; }
  static constexpr bool kHasBias = false;
  __host__ __device__ static constexpr int bias_a_chunk(int) { return 0; }
};

// ---- weight layout of the CTA-pair kernels -------------------------------------------------------------------
// The chain kernels run as CTA pairs (cluster of 2): one M = 256 tcgen05.mma per K = 16 covers a 128-sample tile
// in EACH CTA, and each CTA holds only HALF of the weight rows (N/2), so per SM the L2 -> smem weight traffic and
// the B-operand smem reads are halved.  Stages are K = 64 wide (four MMAs per full/empty barrier round) and every
// (stage, CTA) piece is contiguous in the blob, so a stage is ONE bulk copy per CTA:
//   step s: [stage 0: cta0 piece | cta1 piece][stage 1: ...] ... [bias stage: cta0 | cta1]
//   piece = [k/8 chunks][N/2 rows][8]   (k = 64, or the 32-wide tail of the direction encoding, or 16 for the bias)
constexpr int kPairK = 64;
constexpr int kNumStages2 = 4;
constexpr int kStageBytes2 = 128 * kPairK * 2;     // 16 KB ring slot (N/2 <= 128 rows)
template <class Prog>
struct PairLayout {
  __host__ __device__ static constexpr int ktot(int s) { return (Prog::nk_h(s) + Prog::nk_x(s)) * kKStage; }
  __host__ __device__ static constexpr int kh(int s) { return Prog::nk_h(s) * kKStage; }      // K fed by hs, rest by xs
  __host__ __device__ static constexpr int n_data(int s) { return (ktot(s) + kPairK - 1) / kPairK; }
  __host__ __device__ static constexpr int n_stages(int s) { return n_data(s) + (Prog::kHasBias ? 1 : 0); }
  __host__ __device__ static constexpr int stage_k(int s, int i) {
    return i < n_data(s) ? (ktot(s) - i * kPairK < kPairK ? ktot(s) - i * kPairK : kPairK) : 16;
  }
  // bytes of ONE CTA's piece: (k/8 chunks) x (N/2 rows) x 16 B
  __host__ __device__ static constexpr int piece_bytes(int s, int i) { return stage_k(s, i) * Prog::N(s); }
  __host__ __device__ static constexpr int step_bytes(int s) {
    return 2 * Prog::N(s) * (ktot(s) + (Prog::kHasBias ? 16 : 0));
  }
  __host__ __device__ static constexpr int blob_off(int s) {
    int off = 0;
    for (int i = 0; i < s; ++i) off += step_bytes(i);
    return off;
  }
  // offset of stage i of step s (CTA 0's piece; CTA 1's follows at + piece_bytes) relative to blob_off(s)
  __host__ __device__ static constexpr int stage_off(int s, int i) { return 2 * Prog::N(s) * (i < n_data(s) ? i * kPairK : ktot(s)); }
  static constexpr int kBytes = blob_off(Prog::kSteps);
};

// ---- packed weight buffer ------------------------------------------------------------------------------------
// [fp32 folded kernel W' + bias][fp32 folded heads][forward blob][dgrad blob].
constexpr int kFoldOff = 0;                                  // fp32 W' = W_f W_g[:256] [256,128], then its bias [128]
constexpr int kFoldFloats = 256 * 128 + 128;                 //   (tc_finish_kernel: the rgb kernel's gradient)
constexpr int kHeadOff = kFoldOff + kFoldFloats * 4;         // fp32 [289][4]: row k < 256 (W'''[k], w_s[k]), 256 + i
constexpr int kHeadRows = 289;                               //   (D[i], 0), 288 (b''', b_s) -- the B operands of forward
constexpr int kHeadFloats = 320 * 4;                         //   step 8 and dgrad step 0 (padded: the blobs start
constexpr int kFwdPairOff = kHeadOff + kHeadFloats * 4;      //   128-byte aligned)
constexpr int kBwdPairOff = kFwdPairOff + PairLayout<FwdProg>::kBytes;
constexpr int kPackedBytes = kBwdPairOff + PairLayout<BwdProg>::kBytes;

struct TcParams {
  int64_t w_off[12], b_off[12];   // float offsets into the flat Keras-order parameter buffer, by CHAIN layer (0..7 hidden,
                                  // 8..11 sigma / features / rgb_features / rgb); -1 = an identity layer of the embedding
                                  // (api.cu tc_chain_map): kernel I, bias 0, gradients not flushed
  int x5;                         // chain layer 5 takes the [h, x] concat (else its encoding rows are zero)
  int U;                          // dense_units of the model (even, <= 256): kernels are [fan_in, U] in the flat buffer (the
                                  // rgb_features kernel [U + dd, U/2]); in the chain's 256-wide operands the columns / rows >= U
                                  // are zero -- their activations are relu(0) = 0 -- and are never flushed
  int dx, dd;                     // widths of the encodings the model uses: 3 + 6 L_xyz <= 63, 3 + 6 L_dir <= 27.  PE_L is a
                                  // prefix of PE_10 / PE_4 (utils.py:176-186 appends one sin / cos block per frequency), so a
                                  // model with fewer frequencies runs on the same kernels: the operand keeps all 63 / 27
                                  // columns, the packed weights of the unused ones are zero and their gradients are not flushed
};

// ---- per-tile records in the training workspace (chunk-major bf16) -------------------------------------------
// activations saved by the forward:
constexpr int kRecXS = 0;                          // PE(xyz)      [8 chunks][128][8]   16 KB
constexpr int kRecDS = 16384;                      // PE(dir)      [4 chunks][128][8]    8 KB (the next 8 KB are unused)
constexpr int kRecH0 = 32768;                      // h0..h7       8 x 64 KB
// (the rgb_features activations G are NOT saved: G = h7 W' + PE(dir) W_g[256:] + b' is linear in records that are saved
//  anyway, so the rgb kernel's gradient G^T d(rgb_pre) = W'^T (h7^T d(rgb_pre)) + W_g[256:]^T (PE(dir)^T d(rgb_pre))
//  + b' (x) sum d(rgb_pre) comes from three columns the weight-gradient kernel computes anyway -- tc_finish_kernel)
constexpr int kRecMask = kRecH0 + 8 * kHSBytes;    // ReLU' bits of h0..h7: 8 x [2 halves][128 rows][4 groups] u32 = 32 KB
constexpr int kMaskLayerBytes = 4096;              //   word (h, r, g): columns h*128 + g*32 + (0..31) of row r (one 16-byte
                                                   //   vector per thread of the epilogues);
                                                   //   bit 8 t + q = column 4 q + t (q = 0..7, t = 0..3): byte t holds one
                                                   //   column of every group of four, so that a shift by 7 - q parks the
                                                   //   four flags of columns 4q..4q+3 in the byte msbs, where one prmt with
                                                   //   sign replication expands them to byte / half-word masks (dgrad)
constexpr int kRecBytes = kRecMask + 8 * kMaskLayerBytes;   // 576 KB per 128 samples
// pre-activation gradients written by the dgrad kernel for the weight-gradient GEMMs:
constexpr int kDzZ0 = 0;                           // dZ0..dZ7     8 x 64 KB
constexpr int kDzG = 8 * kHSBytes;                 // (unused since round 2: d rgb_features stays on chip)
constexpr int kDzP = kDzG + 32768;                 // (d rgb_pre[3], d sigma_pre, 0...) [2 chunks][128][8]  4 KB
constexpr int kDzBytes = kDzP + 4096;              // 548 KB per 128 samples
// ---- fp8 records (KNERF_REC_FP8) ---------------------------------------------------------------------------------
// The same records at one byte per element: [features/16 chunks][128 samples][16 B] -- read along the other axis the
// canonical MN-major 8-bit UMMA operand (tc_ptx.cuh), consumed by kind::f8f6f4 MMAs (K = 32 samples each).  Activations
// and encodings are e4m3 at scale 1 (|PE| <= ~6, post-ReLU activations of this network stay orders of magnitude below
// the format's 448); the pre-activation gradients are e5m2 times ONE power-of-two scale per backward call, chosen from
// max|d_pre| (kXOffAmax) so that it lands in [32, 64): e5m2 then has a factor 896 of head room above it and 2^-22 of it
// below.  Both operand roundings are unbiased and independent per element, so they average out over the samples of a
// gradient like the bf16 operand rounding does (measured: +0.4 % relative error of dW_0 at 98k samples, DESIGN.md §4).
// Only the weight-gradient GEMMs see them: the forward and the dgrad chain keep their bf16 operands on chip.
constexpr int kH8Bytes = kTileM * kU;              // 32 KB: one [128 x 256] fp8 record
constexpr int kRec8XS = 0;                         // PE(xyz)  [4 chunks][128][16]   8 KB
constexpr int kRec8DS = 8192;                      // PE(dir)  [2 chunks][128][16]   4 KB (the next 4 KB are unused)
constexpr int kRec8H0 = 16384;                     // h0..h7   8 x 32 KB
constexpr int kRec8Mask = kRec8H0 + 8 * kH8Bytes;  // ReLU' bits, as above (32 KB)
constexpr int kRec8Bytes = kRec8Mask + 8 * kMaskLayerBytes;   // 304 KB per 128 samples
constexpr int kDz8Z0 = 0;                          // dZ0..dZ7 8 x 32 KB
constexpr int kDz8P = 8 * kH8Bytes;                // (d rgb_pre[3], d sigma_pre, 0 x 12) [1 chunk][128][16]  2 KB
constexpr int kDz8Bytes = kDz8P + 2048;            // 258 KB per 128 samples
constexpr int kDz8Top = 6;                         // max|d_pre| * scale lies in [2^(kDz8Top-1), 2^kDz8Top)

// fp32 scratch at the head of the training workspace (zeroed by every backward call): the weight-gradient kernel's
// work-item counter (a uint32), Y = h7^T d(rgb_pre) [256 x 4], Yd = PE(dir)^T d(rgb_pre) [32 x 4] and sum d(rgb_pre) [4]
// -- the rank-3 factors of every gradient that contains d(rgb_features) (tc_finish_kernel).  The counter lies below
// kXOffS: a weight-gradient-only call over fp8 records zeroes only [0, kXOffS).
constexpr int kXOffQueue = 0;
constexpr int kXOffY = 4;
constexpr int kXOffYd = kXOffY + 256 * 4;
constexpr int kXOffS = kXOffYd + 32 * 4;
constexpr int kXOffT = kXOffS + 4;           // T[j][c] = sum_n W_g[j][n] W_c[n][c]                      [256 x 4]
constexpr int kXOffU = kXOffT + 256 * 4;     // U[j][c] = sum_i W_f[i][j] Y[i][c] + b_f[j] s3[c]            [256 x 4]
constexpr int kXOffAmax = kXOffU + 256 * 4;  // fp8 records: bits of max|d_pre| of this call (atomicMax on the uint pattern)
constexpr int kXFloats = kXOffAmax + 4;      // (T, U: written by tc_finish_prep_kernel, read by tc_finish_kernel)
constexpr int kXBytes = ((kXFloats * 4 + 255) / 256) * 256;

// scale of the e5m2 gradient records from the bits of max|d_pre|: 2^(kDz8Top - e) with max = m 2^e, m in [0.5, 1)
__host__ __device__ inline float dz8_scale(uint32_t amax_bits, bool inverse) {
  int e = (int)((amax_bits >> 23) & 0xff) - 126;
  if (amax_bits == 0u || e < -100) e = -100;       // all-zero gradients (or denormal ones): any finite scale will do
  if (e > 100) e = 100;
  const int k = inverse ? e - kDz8Top : kDz8Top - e;
  union { uint32_t u; float f; } c;
  c.u = (uint32_t)(127 + k) << 23;
  return c.f;
}

struct ChainSmem {
  uint8_t hs[2][kHSBytes];
  uint8_t xs[2][kXSBytes];
  uint8_t stage[kNumStages2][kStageBytes2];
  uint64_t full[kNumStages2], empty[kNumStages2], a_ready[2], acc_ready[2], st_ready[2], st_done[2];
  uint32_t tmem_base;
  uint32_t items_issued;      // ordered mode: ring items whose MMAs have been issued (the two issuers take turns)
  uint32_t first_issued[2];   // unordered mode, per tile slot: GEMM steps whose first (accumulate = 0) MMA is issued
};

}  // namespace tcl
}  // namespace knerf
