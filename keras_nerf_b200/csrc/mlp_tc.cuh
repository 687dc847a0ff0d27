// tcgen05 / TMEM / TMA (bf16) MLP path: interface used by api.cu and pipeline.cu
#pragma once
#include "common.cuh"

namespace knerf {

bool tc_path_compiled();
int64_t tc_workspace_bytes(const Model& m, int64_t rows, bool training, bool rec8 = false);   // -1: shape unsupported
int64_t tc_packed_weight_bytes(const Model& m);
int tc_pack_weights(const Model& m, const float* params, void* packed, cudaStream_t st);
// (o,d,t) -> rgbsigma[R*S,4]; training keeps activations in ws.  ordered: the two MMA-issuing threads hand over in
// ring order at inference too (KNERF_TC_ORDERED; training kernels always do)
int tc_forward(const Model& m, const float* params, const void* packed, const float* o, const float* d,
               const float* t, int64_t R, int S, bool training, bool ordered, bool rec8, float* rgbsigma, char* ws,
               int64_t ws_bytes, cudaStream_t st);
// parts: bit 0 = dgrad chain kernel, bit 1 = weight-gradient kernels (3 = the whole backward)
// rec8 (KNERF_REC_FP8; forward and backward of one step must agree): the saved records are fp8 (tc_layout.cuh)
int tc_backward(const Model& m, const float* params, const void* packed, const float* d_pre, int64_t R, int S,
                float* grads, char* ws, int64_t ws_bytes, int parts, bool rec8, cudaStream_t st);

int tc_debug_timing(unsigned long long* host_out, int n);
int tc_debug_wgrad_timing(unsigned long long* host_out, int n);
int tc_debug_dgrad_timing(unsigned long long* host_out, int n);

}  // namespace knerf
