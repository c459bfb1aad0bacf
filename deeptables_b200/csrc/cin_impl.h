// Internal interface between cin_api.cu and the two CIN implementations.
#pragma once
#include <cuda_runtime.h>
#include "cin_shapes.h"

namespace dtb {

size_t cin_fp32_saved_bytes(const CinShape& s, int B);
size_t cin_fp32_workspace_bytes(const CinShape& s, int B, int training);
int cin_fp32_fwd(const CinShape& s, const int32_t* idx, const float* table, const int64_t* row_offsets,
                 const float* weights, const float* bias, float* pooled, void* saved, void* workspace,
                 size_t workspace_bytes, int B, int act, int* status, cudaStream_t st);
int cin_fp32_bwd(const CinShape& s, const int32_t* idx, const float* table, const int64_t* row_offsets,
                 const float* weights, const float* d_pooled, const void* saved, float* grad_table,
                 float* d_weights, float* d_bias, void* workspace, size_t workspace_bytes, int B, int act,
                 cudaStream_t st);

bool cin_tc_supported(const CinShape& s);
bool cin_tc_f16_auto(const CinShape& s);     // precision "auto" resolves to the single-pass fp16 kernels for this shape
size_t cin_tc_saved_bytes(const CinShape& s, int B);
size_t cin_tc_workspace_bytes(const CinShape& s, int B, int training);
// n_pass: 3 = bf16x3 split (fp32-grade), 1 = single pass; f16: single pass on scaled fp16 operands (n_pass must be 1),
// on the cin_tc2.cu kernels or DTB_ERR_UNSUPPORTED when the shape is outside them
int cin_tc_fwd(const CinShape& s, const int32_t* idx, const float* table, const int64_t* row_offsets,
               const float* weights, const float* bias, float* pooled, void* saved, void* workspace,
               size_t workspace_bytes, int B, int act, int n_pass, int f16, int* status, cudaStream_t st);
int cin_tc_bwd(const CinShape& s, const int32_t* idx, const float* table, const int64_t* row_offsets,
               const float* weights, const float* d_pooled, const void* saved, float* grad_table,
               float* d_weights, float* d_bias, void* workspace, size_t workspace_bytes, int B, int act,
               int n_pass, int f16, int phase, cudaStream_t st);

}  // namespace dtb
