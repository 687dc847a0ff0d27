// a6 (KNERF_BF16 mode): the NeRF MLP on Blackwell tensor cores -- tcgen05.mma with TMEM accumulators, weights
// streamed by TMA bulk copies, positional encoding fused into the first-layer prologue and the sigma / rgb
// heads into the epilogue, so per-sample activations never round-trip through HBM at inference
// (keras_nerf/model/nerf/mlp.py:29-50 + keras_nerf/model/nerf/utils.py:176-210).
//
// 256-wide models of up to eight layers with at most one skip concat, L_xyz <= 10, L_dir <= 4 (csrc/api.cu tc_chain_map,
// tc_layout.cuh TcParams); the Python shim runs other shapes in the fp32_tc mode.
//
// Forward kernel (persistent CTA pairs, 384 threads per CTA; roles in tc_roles.cuh):
//   warp 0      TMA producer: streams this CTA's half of the pre-packed bf16 weight blob, K = 64 stages, 4-slot ring
//   warps 1,11  MMA issuers (leader CTA): tcgen05.mma.cta_group::2 (M = 256, N = 256|16, K = 16), alternate items
//   warps 2-9   compute:      PE prologue, TMEM -> register epilogues (ReLU, bf16 pack) that write the next layer's
//                             A operand straight into shared memory, output (sigmoid / ReLU of the head columns).
//                             Biases ride in the GEMM (constant-1 column, tc_layout.cuh); the last step's N = 16
//                             columns are the folded heads' pre-activations (rgb, sigma).
//   warp 10     record store (training): bulk copies of the operand tiles to HBM
// Each CTA keeps TWO 128-sample tiles in flight (accumulators in TMEM columns [0,256) and [256,512)): while
// the tensor core runs tile 1's layer, the compute warps drain tile 0's accumulator and build its next A
// operand, and vice versa.
// Shared memory: 2 x 64 KB hidden activations + 2 x 16 KB encodings + 4 x 16 KB weight stages = 224 KB.
#include "mlp_tc.cuh"

#include <cstdlib>
#include <type_traits>

#include "tc_roles.cuh"

namespace knerf {
using namespace tc;
using namespace tcl;

namespace {

// ---- weight packing --------------------------------------------------------------------------------------
// B operand element of forward step s < 8 at reduction index k (hs part first, then the encoding part), output n
__device__ __forceinline__ float fwd_weight(const float* __restrict__ params, const TcParams& P, int s, int k, int n) {
  const int L = s, kh = FwdProg::nk_h(s) * kKStage, U = P.U;
  if (P.w_off[L] < 0) return (k < kh && k == n) ? 1.f : 0.f;   // identity layer of the embedding
  if (n >= U) return 0.f;
  int row;                                                      // row of the model's kernel [fan_in, U]
  if (k < kh) {
    if (k >= U) return 0.f;
    row = k;
  } else {
    const int j = k - kh;                                       // encoding column
    if (j >= P.dx || (L != 0 && !(L == 5 && P.x5))) return 0.f;
    row = (kh > 0 ? U : 0) + j;
  }
  return params[P.w_off[L] + (int64_t)row * U + n];
}
// W' = W_f W_g[:256] [256,128] and its bias b_f W_g[:256] + b_g [128] in fp32 (tc_layout.cuh), one thread per element,
// and the folded heads (kHeadOff): head row k = (row k of [W'; D; b'] times W_c, then + b_c for the bias row; sigma's
// kernel / bias in column 3).  Block k: k < 256 row k of W', 256 + i row i of W_g[U:] (i < dd), 288 the bias row.
// The products over n run through one fixed reduction tree: the same bits run after run, and zero-padded rows and
// columns (a narrower model embedded in the 256-wide chain) only add exact zeros.
__global__ void __launch_bounds__(128) fold_kernel(const float* __restrict__ params, TcParams P, float* __restrict__ fold,
                                                   float* __restrict__ head) {
  const int U = P.U, H = P.U / 2;
  const float* Wf = params + P.w_off[9];    // features      [U, U]
  const float* Wg = params + P.w_off[10];   // rgb_features  [U + dd, U/2]
  const float* Wc = params + P.w_off[11];   // rgb           [U/2, 3]
  const int n = threadIdx.x, k = blockIdx.x;
  float acc = 0.f;
  if (k < 256 || k == 288) {
    if (n < H && (k < U || k == 288)) {
      const float* row = k < 256 ? Wf + (int64_t)k * U : params + P.b_off[9];
      acc = k < 256 ? 0.f : params[P.b_off[10] + n];
#pragma unroll 8
      for (int j = 0; j < U; ++j) acc = fmaf(row[j], Wg[j * H + n], acc);
    }
    fold[(k < 256 ? k : 256) * 128 + n] = acc;
  } else if (n < H && k - 256 < P.dd) {
    acc = Wg[(int64_t)(U + k - 256) * H + n];
  }
  __shared__ float red[4][3];
  float c3[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    c3[c] = n < H ? acc * Wc[n * 3 + c] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c3[c] += __shfl_xor_sync(0xffffffffu, c3[c], o);
    if ((n & 31) == 0) red[n >> 5][c] = c3[c];
  }
  __syncthreads();
  if (n < 3) {
    float v = (red[0][n] + red[1][n]) + (red[2][n] + red[3][n]);
    if (k == 288) v += params[P.b_off[11] + n];
    head[k * 4 + n] = v;
  } else if (n == 3) {
    head[k * 4 + 3] = k < U ? params[P.w_off[8] + k] : (k == 288 ? params[P.b_off[8]] : 0.f);   // sigma [U, 1], b_s
  }
}
// last forward step: reduction index k (h7, then the direction encoding), output column n.  Column c < 4 takes the bf16
// rounding of head value c, column 4 + c the bf16 rounding of what that leaves: the epilogue adds the two accumulators,
// so the folded weights enter with ~2^-17 relative error instead of one bf16 rounding of the whole product W' W_c
// (which on trained weights, where the terms of W' W_c add up coherently, doubled the fine pass's pixel error).
__device__ __forceinline__ float fold_split(float v, int n) {
  const float hi = bf16_lo(pack_bf16x2(v, 0.f));
  return n < 4 ? hi : v - hi;
}
__device__ __forceinline__ float fold_weight(const float* __restrict__ head, int k, int n) {
  return n < 8 ? fold_split(head[k * 4 + (n & 3)], n) : 0.f;
}
__device__ __forceinline__ float fold_bias(const float* __restrict__ head, int n) {
  return n < 8 ? fold_split(head[288 * 4 + (n & 3)], n) : 0.f;
}
// B operand element of dgrad step b: output n = input feature of the layer (< 256), reduction index k = its output
// feature.  b = 0 goes from (d rgb_pre, d sigma_pre) straight to d(h7): [W''' | w_s][n][k]
__device__ __forceinline__ float bwd_weight(const float* __restrict__ params, const TcParams& P,
                                            const float* __restrict__ head, int b, int k, int n) {
  if (b == 0) return k < 4 ? head[n * 4 + k] : 0.f;
  if (P.w_off[BwdProg::layer(b)] < 0) return n == k ? 1.f : 0.f;   // identity layer of the embedding
  return (n < P.U && k < P.U) ? params[P.w_off[BwdProg::layer(b)] + (int64_t)n * P.U + k] : 0.f;
}

template <class Prog, bool FWD>
__device__ __forceinline__ void pack_pair(const float* __restrict__ params, const TcParams& P,
                                          const float* __restrict__ head, uint8_t* __restrict__ blob, int gtid, int gsz) {
  using PL = PairLayout<Prog>;
  auto weight = [&](int s, int k, int n) -> float {
    if (!FWD) return bwd_weight(params, P, head, s, k, n);
    return s == 8 ? fold_weight(head, k, n) : fwd_weight(params, P, s, k, n);
  };
  for (int v = gtid; v < PL::kBytes / 16; v += gsz) {
    const int byte = v * 16;
    int s = 0;
    while (s + 1 < Prog::kSteps && byte >= PL::blob_off(s + 1)) ++s;
    const int local = byte - PL::blob_off(s);
    const int N = Prog::N(s), half = N / 2, ktot = PL::ktot(s);
    uint32_t w[4] = {0u, 0u, 0u, 0u};
    if (local < 2 * N * ktot) {
      const int i = local / (2 * N * kPairK);                 // stage
      const int rem = local - i * (2 * N * kPairK);
      const int pb = PL::piece_bytes(s, i);
      const int cta = rem / pb, r2 = rem - cta * pb;
      const int c = r2 / (half * 16), nl = (r2 - c * half * 16) / 16;
      const int k0 = i * kPairK + c * 8, n = cta * half + nl;
#pragma unroll
      for (int e = 0; e < 4; ++e) w[e] = pack_bf16x2(weight(s, k0 + 2 * e, n), weight(s, k0 + 2 * e + 1, n));
    } else {   // bias piece [2 chunks][N/2][8]: k = 15 <- bias[n]
      const int rem = local - 2 * N * ktot, pb = 16 * N;
      const int cta = rem / pb, r2 = rem - cta * pb;
      const int cb = r2 / (half * 16), nl = (r2 - cb * half * 16) / 16;
      if (cb == 1)
        w[3] = pack_bf16x2(0.f, s == 8 ? fold_bias(head, cta * half + nl)
                                       : ((P.b_off[s] < 0 || cta * half + nl >= P.U) ? 0.f : params[P.b_off[s] + cta * half + nl]));
    }
    *reinterpret_cast<uint4*>(blob + byte) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

__global__ void __launch_bounds__(256) pack_kernel(const float* __restrict__ params, TcParams P,
                                                   uint8_t* __restrict__ packed) {
  const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
  const float* head = reinterpret_cast<const float*>(packed + kHeadOff);   // written by fold_kernel
  pack_pair<FwdProg, true>(params, P, head, packed + kFwdPairOff, gtid, gsz);
  pack_pair<BwdProg, false>(params, P, head, packed + kBwdPairOff, gtid, gsz);
}

// ---- positional encoding into an A operand -----------------------------------------------------------------
// thread (row r, half h) of the 256 compute threads builds 32 consecutive columns of its row in registers and
// writes them as four 16-byte vectors (512 contiguous bytes per warp and chunk: conflict-free), to the smem
// operand and -- when training -- to the tile's record in HBM.
//
// sin/cos(2^f x): ONE sin/cos pair per coordinate at the half's base frequency (|arg| <= ~100, fast_sincos),
// then angle doubling  sin 2a = 2 sin a cos a,  cos 2a = 1 - 2 sin^2 a.  The absolute error doubles per step
// (<= 32 x 6e-8 after five), far below the bf16 rounding of the operand (2^-9 relative).
// sin/cos for |x| <= a few hundred: two-term Cody-Waite reduction to [-pi, pi] (k * 2pi_hi is exact for |k| < 2^8:
// 2pi_hi has 16 significant bits), then the MUFU units (absolute error ~4e-7 on the reduced range).  ~8
// instructions instead of the ~80 of the full-range sincosf.
__device__ __forceinline__ void fast_sincos(float x, float* sn, float* cs) {
  const float k = rintf(x * 0.15915494309189535f);
  float r = fmaf(k, -6.28314208984375f, x);          // 2pi_hi = 0x40C90F00
  r = fmaf(k, -4.321663826704025e-05f, r);           // 2pi - 2pi_hi
  *sn = __sinf(r);
  *cs = __cosf(r);
}

__device__ __forceinline__ void angle_double(float (&sn)[3], float (&cs)[3]) {
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float s2 = 2.f * sn[c] * cs[c];
    cs[c] = fmaf(-2.f * sn[c], sn[c], 1.f);
    sn[c] = s2;
  }
}

// (REC8: the record is fp8 -- 16 columns per 16-byte vector, chunk index = chunk0 / 2 -- the operand stays bf16)
template <bool REC8>
__device__ __forceinline__ void store_cols(uint8_t* xs, uint8_t* rec, int r, int chunk0, const float* v, int nchunks) {
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (k < nchunks) {
      const uint4 pk = make_uint4(pack_bf16x2(v[8 * k], v[8 * k + 1]), pack_bf16x2(v[8 * k + 2], v[8 * k + 3]),
                                  pack_bf16x2(v[8 * k + 4], v[8 * k + 5]), pack_bf16x2(v[8 * k + 6], v[8 * k + 7]));
      const int off = (chunk0 + k) * kChunkA + r * 16;
      *reinterpret_cast<uint4*>(xs + off) = pk;
      if (!REC8 && rec) *reinterpret_cast<uint4*>(rec + off) = pk;
    }
  }
  if (REC8 && rec) {
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (2 * k < nchunks) {
        const float* x = v + 16 * k;
        const uint4 q = make_uint4(pack_e4m3x4(x[0], x[1], x[2], x[3]), pack_e4m3x4(x[4], x[5], x[6], x[7]),
                                   pack_e4m3x4(x[8], x[9], x[10], x[11]), pack_e4m3x4(x[12], x[13], x[14], x[15]));
        __stcs(reinterpret_cast<uint4*>(rec + ((chunk0 >> 1) + k) * kChunkA + r * 16), q);
      }
    }
  }
}

// PE_10(o + d t) -> 63 columns + the constant-1 column 63 (carries the folded bias, tc_layout.cuh).
// Column order (utils.py:176-186): x y z, then per frequency f: sin(2^f xyz), cos(2^f xyz).
// h = 0: columns 0..31 (identity, f = 0..3, f = 4 up to cos y);  h = 1: columns 32..63 (cos(2^4 z), f = 5..9, 1).
// ray origin, direction and depth of one sample: loaded EARLY (start of the epilogue that precedes the encoding) so
// that the global-memory latency hides behind that epilogue
// (no local memory anywhere in these kernels: with 227 KB of shared memory the SM has no L1 left, a spill or a
// by-reference struct would be an L2 round trip)
__device__ __forceinline__ void load_sample(float (&p)[3], const float* __restrict__ o, const float* __restrict__ d,
                                            const float* __restrict__ t, int64_t g, int64_t M, int S) {
  p[0] = p[1] = p[2] = 0.f;
  if (g < M) {
    const uint32_t ray = (uint32_t)g / (uint32_t)S;   // M < 2^31 (checked by the launcher)
    const float tt = __ldg(t + g);
#pragma unroll
    for (int c = 0; c < 3; ++c) p[c] = __fadd_rn(__ldg(o + ray * 3 + c), __fmul_rn(__ldg(d + ray * 3 + c), tt));   // utils.py:193-196
  }
}
__device__ __forceinline__ void load_dir(float (&x)[3], const float* __restrict__ d, int64_t g, int64_t M, int S) {
  x[0] = x[1] = x[2] = 0.f;
  if (g < M) {
    const uint32_t ray = (uint32_t)g / (uint32_t)S;
#pragma unroll
    for (int c = 0; c < 3; ++c) x[c] = __ldg(d + ray * 3 + c);
  }
}

template <bool REC8>
__device__ __noinline__ void pe_xyz(uint8_t* xs, uint8_t* rec, int r, int h, float px, float py, float pz) {
  const float p[3] = {px, py, pz};
  float sn[3], cs[3], v[34];
#pragma unroll
  for (int c = 0; c < 3; ++c) fast_sincos(h ? 16.f * p[c] : p[c], &sn[c], &cs[c]);
  if (h == 0) {
#pragma unroll
    for (int c = 0; c < 3; ++c) v[c] = p[c];
#pragma unroll
    for (int i = 0; i < 5; ++i) {
#pragma unroll
      for (int c = 0; c < 3; ++c) { v[3 + 6 * i + c] = sn[c]; v[6 + 6 * i + c] = cs[c]; }   // v[32] = cos(2^4 z): h = 1's
      angle_double(sn, cs);
    }
  } else {
    v[0] = cs[2];
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      angle_double(sn, cs);
#pragma unroll
      for (int c = 0; c < 3; ++c) { v[1 + 6 * i + c] = sn[c]; v[4 + 6 * i + c] = cs[c]; }
    }
    v[31] = 1.f;
  }
  store_cols<REC8>(xs, rec, r, 4 * h, v, 4);
}

// PE_4(d) -> 27 columns, zeros in 27..30, the constant-1 column 31 (folded bias of steps 6..9) into chunks 0..3
// of the xs buffer.  h = 0: columns 0..15 (identity, f = 0, 1, sin(4 x));  h = 1: columns 16..31.
// (the record keeps only these 4 chunks: the weight-gradient kernel fetches 8 KB for this operand)
template <bool REC8>
__device__ __noinline__ void pe_dir(uint8_t* xs, uint8_t* rec, int r, int h, float x0, float x1, float x2) {
  const float x[3] = {x0, x1, x2};
  float sn[3], cs[3], v[18];
#pragma unroll
  for (int c = 0; c < 3; ++c) fast_sincos(h ? 4.f * x[c] : x[c], &sn[c], &cs[c]);
  if (h == 0) {
#pragma unroll
    for (int c = 0; c < 3; ++c) v[c] = x[c];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
#pragma unroll
      for (int c = 0; c < 3; ++c) { v[3 + 6 * i + c] = sn[c]; v[6 + 6 * i + c] = cs[c]; }
      angle_double(sn, cs);
    }
    v[15] = sn[0];
  } else {
    v[0] = sn[1]; v[1] = sn[2]; v[2] = cs[0]; v[3] = cs[1]; v[4] = cs[2];
    angle_double(sn, cs);
#pragma unroll
    for (int c = 0; c < 3; ++c) { v[5 + c] = sn[c]; v[8 + c] = cs[c]; }
    v[11] = v[12] = v[13] = v[14] = 0.f;
    v[15] = 1.f;
  }
  store_cols<REC8>(xs, rec, r, 2 * h, v, 2);
}

// ---- epilogue of a hidden step: accumulator -> bf16 A operand of the next step ---------------------------------
// Thread (row r, half h) converts 128 of the 256 columns, 32 at a time.  The bias is already in the accumulator
// (folded into the GEMM), ReLU (mlp.py:33-34) is fused into the bf16 conversion.  mask_out (training): the ReLU'
// bits of the tile, 1 bit per activation (tc_layout.cuh kRecMask) for the dgrad kernel.
// (__noinline__: one body for all eight layers keeps the kernel below the I-cache thrash point.)
// rec8 (fp8 records): the tile's saved activation record goes to HBM from here, 16 columns per 16-byte vector,
// rounded from the fp32 accumulator -- no copy of the operand tile, no hand-shake with a store warp.
// one 32-column group of epi_hidden: v = the accumulator values (already waited for)
// (returns the ReLU' bits of the 32 columns)
template <bool TRAIN, bool REC8>
__device__ __forceinline__ uint32_t epi_hidden_group(const uint32_t (&v)[32], int gI, uint8_t* __restrict__ hs, int h, int r,
                                                     uint8_t* __restrict__ rec8) {
  const int col0 = h * 128 + gI * 32;
  uint32_t mbits = 0u;
#pragma unroll
  for (int c8 = 0; c8 < 4; ++c8) {
    const float* x = reinterpret_cast<const float*>(&v[c8 * 8]);
    const uint4 pk = make_uint4(pack_bf16x2_relu(x[0], x[1]), pack_bf16x2_relu(x[2], x[3]),
                                pack_bf16x2_relu(x[4], x[5]), pack_bf16x2_relu(x[6], x[7]));
    if (TRAIN) {
      // ReLU' bits (tc_layout.cuh kRecMask).  The packed halves are non-negative, so half + 0x7fff has its msb set
      // exactly when the half is > 0 (no carry between the halves); one prmt with sign replication turns the four
      // flags of a word PAIR into four 0x00 / 0xff bytes, one LOP3 files bit q of every byte: 2 ALU-pipe
      // instructions per pair where HSET2 + LOP3 per word were 4 (forward, training: 1.09 -> 1.04 ns per sample).
      const uint32_t u0 = prmt(pk.x + 0x7fff7fffu, pk.y + 0x7fff7fffu, 0xFDB9u);
      const uint32_t u1 = prmt(pk.z + 0x7fff7fffu, pk.w + 0x7fff7fffu, 0xFDB9u);
      mbits |= u0 & (0x01010101u << (2 * c8));
      mbits |= u1 & (0x01010101u << (2 * c8 + 1));
    }
    // next layer's A operand, in place; with bf16 records also the saved record (stored to HBM by warp 10)
    *reinterpret_cast<uint4*>(hs + ((col0 >> 3) + c8) * kChunkA + r * 16) = pk;
  }
  if (TRAIN && REC8 && rec8 != nullptr) {
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const float* x = reinterpret_cast<const float*>(&v[16 * k]);
      const uint4 q = make_uint4(pack_e4m3x4_relu(x[0], x[1], x[2], x[3]), pack_e4m3x4_relu(x[4], x[5], x[6], x[7]),
                                 pack_e4m3x4_relu(x[8], x[9], x[10], x[11]),
                                 pack_e4m3x4_relu(x[12], x[13], x[14], x[15]));
      __stcs(reinterpret_cast<uint4*>(rec8 + ((col0 >> 4) + k) * kChunkA + r * 16), q);
    }
  }
  return mbits;
}

template <bool TRAIN, bool REC8>
__device__ __noinline__ void epi_hidden(uint32_t tacc, uint8_t* __restrict__ hs, int h, int r,
                                        uint8_t* __restrict__ mask_out, uint8_t* __restrict__ rec8) {
  // (measured and dropped: a second accumulator group in flight, so that the TMEM load of the next 32 columns runs under
  //  the conversion of the current ones, and IMADs instead of integer adds for the flag additions -- no change in the
  //  kernel's time, which at this point moves with the power cap more than with the instruction count)
  uint32_t m0 = 0u, m1 = 0u, m2 = 0u, m3 = 0u;
#pragma unroll 1
  for (int gI = 0; gI < 4; ++gI) {
    uint32_t v[32];
    tmem_ld32_issue(tacc + h * 128 + gI * 32, v);
    tmem_ld32_wait(v);
    const uint32_t mb = epi_hidden_group<TRAIN, REC8>(v, gI, hs, h, r, rec8);
    m0 = gI == 0 ? mb : m0; m1 = gI == 1 ? mb : m1; m2 = gI == 2 ? mb : m2; m3 = gI == 3 ? mb : m3;
  }
  // the thread's 128 ReLU' bits leave as ONE 16-byte store (512 contiguous bytes per warp)
  if (TRAIN && mask_out != nullptr) *reinterpret_cast<uint4*>(mask_out + h * 2048 + r * 16) = make_uint4(m0, m1, m2, m3);
}

// ---- the fused forward kernel ----------------------------------------------------------------------------
// Launched as clusters of 2: the CTA pair shares every weight stage through cta_group::2 MMAs (tc_roles.cuh); a
// work unit is four tiles (two per CTA).
template <bool TRAIN, bool REC8>
__global__ void __launch_bounds__(kThreads, 1)
tc_mlp_fwd_kernel(const uint8_t* __restrict__ packed, const float* __restrict__ o, const float* __restrict__ d,
                  const float* __restrict__ t, int64_t M, int S, float4* __restrict__ rgbsigma,
                  uint8_t* __restrict__ rec, int ordered) {
  using Prog = FwdProg;
  constexpr int kLast = Prog::kSteps - 1;
  constexpr int kRB = REC8 ? kRec8Bytes : kRecBytes, kOffXS = REC8 ? kRec8XS : kRecXS, kOffDS = REC8 ? kRec8DS : kRecDS,
                kOffMask = REC8 ? kRec8Mask : kRecMask;
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
    if (lane == 0) producer_role<Prog>(sm, packed + kFwdPairOff, cta, n_pairs, first, stride);
  } else if (warp == 1) {
    if (lane == 0 && cta == 0) mma_role<Prog>(sm, tmem, 0u, ordered != 0, n_pairs, first, stride);
    else if (lane == 0) relay_role<Prog>(sm, n_pairs, first, stride);   // peer CTA: its warp 1 is otherwise idle
  } else if (warp == 11) {
    if (lane == 0 && cta == 0) mma_role<Prog>(sm, tmem, 1u, ordered != 0, n_pairs, first, stride);
  } else if (warp == 10) {
    // ============== record store (training): the operand tiles h0..h7 -> HBM, bulk copies ======================
    if constexpr (TRAIN && !REC8) {
      if (lane == 0) {
        store_role(sm, 8, n_tiles, n_pairs, first, stride, tile_of,
                   [&](int item, int64_t tile) { return rec + tile * kRecBytes + kRecH0 + item * kHSBytes; },
                   [](int) { return (uint32_t)kHSBytes; });
      }
    }
  } else {
    // =========================== compute warps ==========================
    const int q = warp & 3, h = (warp - 2) >> 2;
    const int r = q * 32 + lane;
    const uint32_t lane_base = (uint32_t)(q * 32) << 16;
    uint32_t acc_par[2] = {0, 0};

    ChainHandshake<TRAIN && !REC8> hk;
    auto prologue = [&](int64_t pair, int tl, const float (&p)[3]) {
      const int64_t tile = tile_of(pair, tl);
      pe_xyz<REC8>(sm.xs[tl], (TRAIN && tile < n_tiles) ? rec + tile * kRB + kOffXS : nullptr, r, h, p[0], p[1], p[2]);
      hk.arrive(sm, tl, lane, false);
    };

    KN_PROF_DECL();
    KN_PROF_BEGIN(t_c);
    if (first < n_pairs) {
#pragma unroll 1
      for (int tl = 0; tl < 2; ++tl) {
        float p0[3];
        load_sample(p0, o, d, t, tile_of(first, tl) * kTileM + r, M, S);
        prologue(first, tl, p0);
      }
    }
    for (int64_t pair = first; pair < n_pairs; pair += stride) {
      for (int s = 0; s < Prog::kSteps; ++s) {
#pragma unroll 1
        for (int tl = 0; tl < 2; ++tl) {
          const int64_t tile = tile_of(pair, tl);
          const int64_t g = tile * kTileM + r;
          const bool valid = g < M;
          const bool save = TRAIN && tile < n_tiles;
          uint8_t* rec_t = rec + tile * kRB;
          KN_PROF_BEGIN(t_w);
          mbar_wait_cluster(&sm.acc_ready[tl], acc_par[tl]);
          KN_PROF_END(t_w, 4);
          KN_PROF_BEGIN(t_e);
          acc_par[tl] ^= 1;
          tc_fence_after();

          if (s < kLast) {
            // hidden layers: 128 of the 256 columns per thread
            float dirv[3];
            if (s == 5) load_dir(dirv, d, g, M, S);   // fetched now, used after the epilogue: the L2 latency hides behind it
            hk.wait_writable(sm, tl);
            epi_hidden<TRAIN, REC8>(tmem + lane_base + tl * 256, sm.hs[tl], h, r,
                                    save ? rec_t + kOffMask + s * kMaskLayerBytes : nullptr,
                                    (REC8 && save) ? rec_t + kRec8H0 + s * kH8Bytes : nullptr);
            if (s == 5) {
              // xs[tl] is dead after layer 5 (skip concat consumed): it now carries PE(dir) for the last step
              pe_dir<REC8>(sm.xs[tl], save ? rec_t + kOffDS : nullptr, r, h, dirv[0], dirv[1], dirv[2]);
            }
            hk.arrive(sm, tl, lane, true);
          } else {
            // columns 0..2 (+ 4..6): the rgb pre-activations, 3 (+ 7): sigma's (heads folded into the step, biases
            // included; mlp.py:40, 43-48).  One half-row thread per row finishes it; the other starts the next tile.
            const int64_t next = pair + stride;
            float nin[3] = {0.f, 0.f, 0.f};   // the next tile of this slot: fetch its sample now, encode it afterwards
            if (next < n_pairs) load_sample(nin, o, d, t, tile_of(next, tl) * kTileM + r, M, S);
            if (h == 0) {   // warp-uniform
              float a[8];
              tmem_ld8(tmem + lane_base + tl * 256, a);
              const float z[4] = {a[0] + a[4], a[1] + a[5], a[2] + a[6], a[3] + a[7]};
              if (valid)
                rgbsigma[g] = make_float4(1.f / (1.f + expf(-z[0])), 1.f / (1.f + expf(-z[1])), 1.f / (1.f + expf(-z[2])),
                                          fmaxf(z[3], 0.f));
            }
            tc_fence_before();
            // this tile is finished: start the next pair's tile in the same slot right away
            if (next < n_pairs) prologue(next, tl, nin);
          }
          KN_PROF_END(t_e, 6 + tl * 16 + s);
        }
      }
    }
    KN_PROF_END(t_c, 5);
    if (tid == 64) { KN_PROF_FLUSH(); }
  }
  chain_teardown(tmem, warp);
}

}  // namespace

bool tc_path_compiled() { return true; }

// diagnostic (-DKNERF_TC_TIMING builds only): copy and clear the forward kernel's per-CTA cycle counters
int tc_debug_timing(unsigned long long* host_out, int n) { return KN_PROF_READ(g_tc_prof, host_out, n); }

int64_t tc_packed_weight_bytes(const Model& m) { return is_flagship(m) ? kPackedBytes : -1; }

int64_t tc_workspace_bytes(const Model& m, int64_t rows, bool training, bool rec8) {
  if (!is_flagship(m)) return -1;
  if (!training) return 256;
  return kXBytes + cdiv(rows, kTileM) * (int64_t)(rec8 ? kRec8Bytes + kDz8Bytes : kRecBytes + kDzBytes) + 256;
}

TcParams tc_make_params(const Model& m) {
  TcParams P;
  int map[8];
  tc_chain_map(m, map);   // (callers have checked is_flagship)
  for (int c = 0; c < 8; ++c) {
    P.w_off[c] = map[c] < 0 ? -1 : m.L[map[c]].w_off;
    P.b_off[c] = map[c] < 0 ? -1 : m.L[map[c]].b_off;
  }
  for (int i = 0; i < 4; ++i) { P.w_off[8 + i] = m.L[m.n_layers + i].w_off; P.b_off[8 + i] = m.L[m.n_layers + i].b_off; }
  P.x5 = (map[5] >= 0 && m.L[map[5]].k_x > 0) ? 1 : 0;
  P.U = m.U;
  P.dx = m.dx;
  P.dd = m.dd;
  return P;
}

int tc_pack_weights(const Model& m, const float* params, void* packed, cudaStream_t st) {
  if (!is_flagship(m)) return fail(KNERF_ERR_UNSUPPORTED, "KNERF_BF16 implements models of dense_units <= 256 (even), up to 8 layers, at most one skip concat (not into the heads), L_xyz <= 10, L_dir <= 4");
  KN_CHECK_ARG((reinterpret_cast<uintptr_t>(packed) & 15) == 0, "tc_pack_weights: packed must be 16-byte aligned");
  fold_kernel<<<kHeadRows, 128, 0, st>>>(params, tc_make_params(m), reinterpret_cast<float*>((uint8_t*)packed + kFoldOff),
                                         reinterpret_cast<float*>((uint8_t*)packed + kHeadOff));
  KN_LAUNCH_CHECK();
  pack_kernel<<<kNumSMs * 2, 256, 0, st>>>(params, tc_make_params(m), (uint8_t*)packed);
  KN_LAUNCH_CHECK();
  return KNERF_OK;
}

int tc_forward(const Model& m, const float* params, const void* packed, const float* o, const float* d, const float* t,
               int64_t R, int S, bool training, bool ordered_issue, bool rec8, float* rgbsigma, char* ws,
               int64_t ws_bytes, cudaStream_t st) {
  (void)params;
  if (!is_flagship(m)) return fail(KNERF_ERR_UNSUPPORTED, "KNERF_BF16 implements models of dense_units <= 256 (even), up to 8 layers, at most one skip concat (not into the heads), L_xyz <= 10, L_dir <= 4");
  const int64_t M = R * S;
  if (training && ws_bytes < tc_workspace_bytes(m, M, true, rec8))
    return fail(KNERF_ERR_WORKSPACE, "tc_forward: workspace %lld < %lld bytes", (long long)ws_bytes,
                (long long)tc_workspace_bytes(m, M, true, rec8));
  KN_CHECK_ARG((reinterpret_cast<uintptr_t>(rgbsigma) & 15) == 0 && (reinterpret_cast<uintptr_t>(packed) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(ws) & 15) == 0,
               "tc_forward: rgbsigma / packed / workspace must be 16-byte aligned");
  KN_CHECK_ARG(M < (int64_t(1) << 31), "tc_forward: at most 2^31 - 1 samples per call");
  // MMA issue order (tc_roles.cuh): bit-reproducible when training, free-running at inference unless the call
  // carries KNERF_TC_ORDERED
  const int ordered = (training || ordered_issue) ? 1 : 0;
  auto kernel = !training ? &tc_mlp_fwd_kernel<false, false>
                : rec8    ? &tc_mlp_fwd_kernel<true, true>
                          : &tc_mlp_fwd_kernel<true, false>;
  return launch_chain(kernel, cdiv(M, kTileM), st, (const uint8_t*)packed, o, d, t, M, S, (float4*)rgbsigma,
                      training ? (uint8_t*)ws + kXBytes : nullptr, ordered);
}

}  // namespace knerf
