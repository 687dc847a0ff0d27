/* knerf_debug.h -- diagnostics of libknerf.so that are NOT part of the drop-in boundary (include/knerf.h).
 * Self-tests that pin the UMMA descriptor encodings (tests/test_gpu_tc.py) and the read-out of the optional
 * in-kernel cycle counters.  None of them changes how any other entry point behaves. */
#ifndef KNERF_DEBUG_H
#define KNERF_DEBUG_H

#include "knerf.h"

#ifdef __cplusplus
extern "C" {
#endif

/* One tcgen05 tile, D[128,N] (fp32, row-major) = A[128,K] * B[N,K]^T from bf16 operand blobs in the library's
 * chunk-major layout ([K/8][rows][8] for mode 0 = K-major; [rows/8][K][8] for mode 1 = MN-major, the
 * weight-gradient form).  mode 2: the MN-major form over fp8 blobs [rows/16][K][16], A = e4m3, B = e5m2
 * (kind::f8f6f4, K = 32 per instruction) -- the weight-gradient GEMM over fp8 records. */
int knerf_selftest_umma(int mode, const void* a_blob, const void* b_blob, int N, int K, float* d_out,
                        void* stream);

/* Same for one tcgen05.mma.cta_group::2 tile pair: D[256,N] = A[256,K] * B[N,K]^T, a_blob = [2][K/8][128][8],
 * b_blob = [2][K/8][N/2][8] (CTA c of the pair owns A rows 128c.. and B rows c*N/2..). */
int knerf_selftest_umma2(const void* a_blob, const void* b_blob, int N, int K, float* d_out, void* stream);

/* Per-CTA clock64() counters of the BF16 forward kernel (40 uint64 per CTA; slots documented in
 * csrc/tc_roles.cuh), copied to host_out and cleared.  Returns the number of values written; 0 unless the
 * library was built with -DKNERF_TC_TIMING (release builds carry no instrumentation). */
int knerf_debug_tc_timing(unsigned long long* host_out, int n);

/* The same for the BF16 dgrad kernel (same 40 slots; slot 15 + 16 tl: its per-tile prologue). */
int knerf_debug_dgrad_timing(unsigned long long* host_out, int n);

/* The same for the BF16 weight-gradient kernel (24 uint64 per CTA; slots documented in csrc/mlp_tc_bwd.cu kWProf):
 * wait and busy cycles of its producer, issuers and flush warps, which arrival released each ring slot last, items
 * and tiles per CTA, %globaltimer at CTA start and end. */
int knerf_debug_wgrad_timing(unsigned long long* host_out, int n);

#ifdef __cplusplus
}
#endif
#endif /* KNERF_DEBUG_H */
