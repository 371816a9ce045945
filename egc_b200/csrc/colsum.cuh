// Deterministic two-stage column sum of a row-major fp32 matrix: out[c] = sum_r in[r, c].
// Used for d_bias = colsum(grad_out) and d_b_comb = colsum(d_lin).  With a gate and / or a scale (the backward of a fused
// ReLU / affine epilogue) each term is first masked and scaled as backward pass 1 does it: (gate[r, c] > 0 ? in : 0) * scale[c].
#pragma once

#include <algorithm>

#include "common.cuh"

namespace egc {

constexpr int kColsumRowsPerCta = 8;   // blockDim = (32, 8)

inline int colsum_slabs(int n_rows) {
  return std::max(1, std::min(sm_count() * 2, ceil_div(n_rows, 64)));
}

inline size_t colsum_workspace_bytes(int n_rows, int n_cols) {
  return static_cast<size_t>(colsum_slabs(n_rows)) * n_cols * sizeof(float) + 256;
}

template <bool EPI>
static __global__ void k_colsum_stage1(const float* __restrict__ in, const float* __restrict__ gate, const float* __restrict__ scale,
                                       int n_rows, int n_cols, int rows_per_slab, float* __restrict__ partial) {
  __shared__ float red[kColsumRowsPerCta][33];
  const int r0 = blockIdx.x * rows_per_slab, r1 = min(r0 + rows_per_slab, n_rows);
  for (int c0 = 0; c0 < n_cols; c0 += 32) {
    const int c = c0 + threadIdx.x;
    float s = 0.f;
    if (c < n_cols) {
      for (int r = r0 + threadIdx.y; r < r1; r += kColsumRowsPerCta) {
        const int64_t i = static_cast<int64_t>(r) * n_cols + c;
        float v = __ldg(in + i);
        if constexpr (EPI) {
          if (gate != nullptr) v = __ldg(gate + i) > 0.f ? v : 0.f;
          if (scale != nullptr) v *= __ldg(scale + c);
        }
        s += v;
      }
    }
    red[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.y == 0 && c < n_cols) {
      float t = 0.f;
#pragma unroll
      for (int y = 0; y < kColsumRowsPerCta; ++y) t += red[y][threadIdx.x];
      partial[static_cast<int64_t>(blockIdx.x) * n_cols + c] = t;
    }
    __syncthreads();
  }
}

// one warp per column: lanes stride over the slabs (fixed order -> deterministic), then a shuffle tree
static __global__ void k_colsum_stage2(const float* __restrict__ partial, int n_slabs, int n_cols, float* __restrict__ out) {
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= n_cols) return;
  float t = 0.f;
  for (int s = lane; s < n_slabs; s += 32) t += partial[static_cast<int64_t>(s) * n_cols + c];
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(kFull, t, o);
  if (lane == 0) out[c] = t;
}

inline int colsum_f32(const float* in, int n_rows, int n_cols, float* out, void* ws, size_t ws_bytes, cudaStream_t st,
                      const float* gate = nullptr, const float* scale = nullptr) {
  EGC_REQUIRE(in && out && ws && n_rows > 0 && n_cols > 0, "colsum: bad arguments");
  EGC_REQUIRE(ws_bytes >= colsum_workspace_bytes(n_rows, n_cols), "colsum: workspace too small");
  const int slabs = colsum_slabs(n_rows);
  const int rows_per_slab = ceil_div(n_rows, slabs);
  float* partial = static_cast<float*>(ws);
  {
    LaunchScope egc_ls_("k_colsum_stage1", st);
    if (gate != nullptr || scale != nullptr)
      k_colsum_stage1<true><<<slabs, dim3(32, kColsumRowsPerCta), 0, st>>>(in, gate, scale, n_rows, n_cols, rows_per_slab, partial);
    else
      k_colsum_stage1<false><<<slabs, dim3(32, kColsumRowsPerCta), 0, st>>>(in, nullptr, nullptr, n_rows, n_cols, rows_per_slab, partial);
  }
  EGC_LAUNCH_CHECK("k_colsum_stage1");
  {
    LaunchScope egc_ls_("k_colsum_stage2", st);
    k_colsum_stage2<<<ceil_div(n_cols, 8), 256, 0, st>>>(partial, slabs, n_cols, out);
  }
  EGC_LAUNCH_CHECK("k_colsum_stage2");
  return EGC_OK;
}

}  // namespace egc
