// Internal interface between the projection entry points (project.cu) and the two kernel
// families: exact-fp32 FFMA tiles (project.cu) and tcgen05 tensor-core tiles (project_tc.cu).
#pragma once

#include "common.cuh"

namespace egc {

// exact-fp32 FFMA tiles (project.cu)
int project_fwd_simt(const float* x, const float* w_bases, const float* w_comb, const float* b_comb, int n, int f_in,
                     int bd, int hab, int sigmoid, float* bases, float* weightings, cudaStream_t st);
size_t project_bwd_simt_workspace(int n, int f_in, int bd, int hab);
int project_bwd_simt(const float* x, const float* w_bases, const float* w_comb, const float* d_bases,
                     const float* d_lin, int n, int f_in, int bd, int hab, float* d_x, float* d_w_bases,
                     float* d_w_comb, float* d_b_comb, void* workspace, size_t workspace_bytes, cudaStream_t st);

// tensor-core (tcgen05, kind::tf32) path; n_terms = 3 -> 3xTF32 split (fp32-level accuracy), 1 -> plain TF32
bool project_tc_supported(int n, int f_in, int bd, int hab);
// the operands and outputs of k_project_tc are read and written in 16-byte pieces: true when every non-NULL pointer is
// 16-byte aligned
bool tc_aligned(const void* a, const void* b, const void* c, const void* d = nullptr);
int project_fwd_tc(const float* x, const float* w_bases, const float* w_comb, const float* b_comb, int n, int f_in,
                   int bd, int hab, int sigmoid, float* bases, float* weightings, int n_terms, cudaStream_t st);
// the same with the basis rows stored as bf16 (round to nearest even); the weightings stay fp32
int project_fwd_tc_bf16(const float* x, const float* w_bases, const float* w_comb, const float* b_comb, int n, int f_in,
                        int bd, int hab, int sigmoid, uint16_t* bases, float* weightings, int n_terms, cudaStream_t st);
int project_fwd_simt_bf16(const float* x, const float* w_bases, const float* w_comb, const float* b_comb, int n, int f_in,
                          int bd, int hab, int sigmoid, uint16_t* bases, float* weightings, cudaStream_t st);
size_t project_bwd_tc_workspace(int n, int f_in, int bd, int hab);
int project_bwd_tc(const float* x, const float* w_bases, const float* w_comb, const float* d_bases, const float* d_lin,
                   int n, int f_in, int bd, int hab, float* d_x, float* d_w_bases, float* d_w_comb, float* d_b_comb,
                   int n_terms, void* workspace, size_t workspace_bytes, cudaStream_t st);

// tensor-core parameter gradients (wgrad_tc.cu): dW_b = x^T d_bases, dW_c = d_lin^T x
bool wgrad_tc_supported(int n, int f_in, int bd, int hab);
size_t wgrad_tc_workspace(int n, int f_in, int bd, int hab);
int wgrad_tc(const float* x, const float* d_bases, const float* d_lin, int n, int f_in, int bd, int hab,
             float* d_w_bases, float* d_w_comb, int n_terms, void* workspace, size_t workspace_bytes, cudaStream_t st);
// deterministic sum of the per-CTA partial tiles [n_cta][128][n_pad]: accumulator column n < n1 -> dW_b[m][n], column
// n2_col0 + j (j < n2) -> dW_c[j][m]
int wgrad_reduce(const float* partial, int n_cta, int f_in, int n1, int n2, int n_pad, int n2_col0, float* d_w_bases,
                 float* d_w_comb, cudaStream_t st);

// the same product with MN-major operands straight from TMA (wgrad_mn.cu): no register transposes
bool wgrad_mn_supported(int n, int f_in, int bd, int hab);
size_t wgrad_mn_workspace(int n, int f_in, int bd, int hab);
int wgrad_mn(const float* x, const float* d_bases, const float* d_lin, int n, int f_in, int bd, int hab,
             float* d_w_bases, float* d_w_comb, int n_terms, void* workspace, size_t workspace_bytes, cudaStream_t st);

}  // namespace egc
