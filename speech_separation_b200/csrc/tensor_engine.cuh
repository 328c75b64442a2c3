// TENSOR engine: tcgen05/TMEM/TMA kernels for the production dimensions.
#pragma once
#include "common.cuh"

namespace vatss {

bool tensor_engine_supports(const vatss_model_desc* d);
const char* tensor_engine_unsupported_reason(const vatss_model_desc* d);   // NULL if supported
size_t tensor_engine_packed_bytes(const vatss_model_desc* d);
size_t tensor_engine_workspace_bytes(const vatss_model_desc* d, int B, int T, int Tv, int L, int S);
int tensor_engine_pack(const vatss_model_desc* d, const float* const* params, void* packed, cudaStream_t st);
int tensor_engine_forward(const vatss_model_desc* d, const float* const* params, const void* packed,
                          const float* mix, const float* emb1, const float* emb2, int B, int T, int Tv, int L,
                          int S, float* s1_pred, float* s2_pred, void* workspace, cudaStream_t st);
// the part of tensor_engine_forward after the last block: x16 = PReLU(x) (B,S,C,N) fp16, enc32 (B,L,N); the workspace
// is carved as tensor_engine_forward carves it for (B, Tv, L, S)
int tensor_engine_tail(const vatss_model_desc* d, const float* const* params, const void* packed, const __half* x16,
                       const float* enc32, int B, int T, int Tv, int L, int S, float* s1_pred, float* s2_pred,
                       void* workspace, cudaStream_t st);

}  // namespace vatss
