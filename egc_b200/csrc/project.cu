// Dense projections of the EGConv layer and their autograd:
//   bases = x . W_b,  weightings = act(x . W_c^T + b_c)          (ref optimized_layers.py:180-184)
// This file holds the exact-fp32 FFMA tile kernel (any shape) and the extern "C" entry points;
// the tcgen05 tensor-core path lives in project_tc.cu and is selected by `algo`.
#include <algorithm>

#include "bf16.cuh"
#include "colsum.cuh"
#include "common.cuh"
#include "project.cuh"

namespace egc {

constexpr int kBM = 128, kBK = 16, kGemmThreads = 256;

// C[M,N] (+)= A_op[M,K] . B_op[K,N]  (+ bias[N]) (sigmoid)
//   A_op(m,k) = A_KCONTIG ? a[m*lda + k] : a[k*lda + m]
//   B_op(k,n) = B_NCONTIG ? b[k*ldb + n] : b[n*ldb + k]
// grid = (ceil(N/BN), ceil(M/BM), splits); with splits > 1 each z-slice reduces its own K range
// into c + z * M * ldc (split-K partials, summed by k_reduce_splits).
// CT = element type of C: float, or bf16 (each result rounded to nearest even; `accumulate` is ignored)
template <int BN, bool A_KCONTIG, bool B_NCONTIG, class CT = float>
__global__ void __launch_bounds__(kGemmThreads) k_gemm_f32(const float* __restrict__ a, int lda,
                                                           const float* __restrict__ b, int ldb,
                                                           CT* __restrict__ c, int ldc, int M, int N, int K,
                                                           int k_per_split, const float* __restrict__ bias,
                                                           int sigmoid, int accumulate) {
  constexpr int TM = 8, TN = BN / 16;
  __shared__ __align__(16) float As[kBK][kBM + 4];
  __shared__ __align__(16) float Bs[kBK][BN + 4];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * kBM, n0 = blockIdx.x * BN;
  const int kb = blockIdx.z * k_per_split, ke = min(K, kb + k_per_split);
  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  for (int k0 = kb; k0 < ke; k0 += kBK) {
    // ---- A tile
    if (A_KCONTIG) {
      const int kk = tid & (kBK - 1), mm0 = tid >> 4;
#pragma unroll
      for (int i = 0; i < kBM / 16; ++i) {
        const int mm = mm0 + i * 16, m = m0 + mm, k = k0 + kk;
        As[kk][mm] = (m < M && k < ke) ? __ldg(a + static_cast<int64_t>(m) * lda + k) : 0.f;
      }
    } else {
      const int mm = tid & (kBM - 1), kk0 = tid >> 7;
#pragma unroll
      for (int i = 0; i < kBK / 2; ++i) {
        const int kk = kk0 + i * 2, m = m0 + mm, k = k0 + kk;
        As[kk][mm] = (m < M && k < ke) ? __ldg(a + static_cast<int64_t>(k) * lda + m) : 0.f;
      }
    }
    // ---- B tile
    if (B_NCONTIG) {
      const int nn = tid % BN, kk0 = tid / BN;
      constexpr int KSTEP = kGemmThreads / BN;
#pragma unroll
      for (int i = 0; i < kBK / KSTEP; ++i) {
        const int kk = kk0 + i * KSTEP, n = n0 + nn, k = k0 + kk;
        Bs[kk][nn] = (n < N && k < ke) ? __ldg(b + static_cast<int64_t>(k) * ldb + n) : 0.f;
      }
    } else {
      const int kk = tid & (kBK - 1), nn0 = tid >> 4;
#pragma unroll
      for (int i = 0; i < BN / 16; ++i) {
        const int nn = nn0 + i * 16, n = n0 + nn, k = k0 + kk;
        Bs[kk][nn] = (n < N && k < ke) ? __ldg(b + static_cast<int64_t>(n) * ldb + k) : 0.f;
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kBK; ++kk) {
      float av[TM], bv[TN];
#pragma unroll
      for (int i = 0; i < TM; i += 4) {
        const float4 t = *reinterpret_cast<const float4*>(&As[kk][ty * TM + i]);
        av[i] = t.x; av[i + 1] = t.y; av[i + 2] = t.z; av[i + 3] = t.w;
      }
#pragma unroll
      for (int j = 0; j < TN; j += 4) {
        const float4 t = *reinterpret_cast<const float4*>(&Bs[kk][tx * TN + j]);
        bv[j] = t.x; bv[j + 1] = t.y; bv[j + 2] = t.z; bv[j + 3] = t.w;
      }
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }

  CT* cz = c + static_cast<int64_t>(blockIdx.z) * M * ldc;
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int m = m0 + ty * TM + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int n = n0 + tx * TN + j;
      if (n >= N) continue;
      float v = acc[i][j];
      CT* dst = cz + static_cast<int64_t>(m) * ldc + n;
      if constexpr (!kBf16<CT>) {
        if (accumulate) v += *dst;
      }
      if (bias != nullptr) v += __ldg(bias + n);
      if (sigmoid) v = 1.f / (1.f + expf(-v));
      if constexpr (kBf16<CT>) *dst = __float2bfloat16_rn(v);
      else *dst = v;
    }
  }
}

__global__ void k_reduce_splits(const float* __restrict__ partial, int splits, int64_t count, float* __restrict__ out) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= count) return;
  float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
  int z = 0;
  for (; z + 4 <= splits; z += 4) {
    t0 += partial[static_cast<int64_t>(z) * count + i];
    t1 += partial[static_cast<int64_t>(z + 1) * count + i];
    t2 += partial[static_cast<int64_t>(z + 2) * count + i];
    t3 += partial[static_cast<int64_t>(z + 3) * count + i];
  }
  for (; z < splits; ++z) t0 += partial[static_cast<int64_t>(z) * count + i];
  out[i] = (t0 + t1) + (t2 + t3);
}

template <bool A_KCONTIG, bool B_NCONTIG, class CT = float>
static int gemm_f32(const float* a, int lda, const float* b, int ldb, CT* c, int ldc, int M, int N, int K,
                    int splits, const float* bias, int sigmoid, int accumulate, cudaStream_t st) {
  const int k_per_split = ceil_div(ceil_div(K, splits), kBK) * kBK;
  LaunchScope ls("k_gemm_f32", st);
  if (N > 64) {
    dim3 grid(ceil_div(N, 128), ceil_div(M, kBM), splits);
    k_gemm_f32<128, A_KCONTIG, B_NCONTIG, CT><<<grid, kGemmThreads, 0, st>>>(a, lda, b, ldb, c, ldc, M, N, K, k_per_split,
                                                                       bias, sigmoid, accumulate);
  } else {
    dim3 grid(ceil_div(N, 64), ceil_div(M, kBM), splits);
    k_gemm_f32<64, A_KCONTIG, B_NCONTIG, CT><<<grid, kGemmThreads, 0, st>>>(a, lda, b, ldb, c, ldc, M, N, K, k_per_split,
                                                                      bias, sigmoid, accumulate);
  }
  EGC_LAUNCH_CHECK("k_gemm_f32");
  return EGC_OK;
}

static int splitk_slabs(int n) { return std::max(1, std::min(sm_count() * 2, ceil_div(n, 256))); }

int project_fwd_simt(const float* x, const float* w_bases, const float* w_comb, const float* b_comb, int n, int f_in,
                     int bd, int hab, int sigmoid, float* bases, float* weightings, cudaStream_t st) {
  // bases[n,bd] = x[n,f_in] . W_b[f_in,bd]
  if (int rc = gemm_f32<true, true>(x, f_in, w_bases, bd, bases, bd, n, bd, f_in, 1, nullptr, 0, 0, st)) return rc;
  // weightings[n,hab] = act(x . W_c[hab,f_in]^T + b_c)
  return gemm_f32<true, false>(x, f_in, w_comb, f_in, weightings, hab, n, hab, f_in, 1, b_comb, sigmoid, 0, st);
}

int project_fwd_simt_bf16(const float* x, const float* w_bases, const float* w_comb, const float* b_comb, int n, int f_in,
                          int bd, int hab, int sigmoid, uint16_t* bases, float* weightings, cudaStream_t st) {
  if (int rc = gemm_f32<true, true, bf16>(x, f_in, w_bases, bd, reinterpret_cast<bf16*>(bases), bd, n, bd, f_in, 1, nullptr, 0, 0, st))
    return rc;
  return gemm_f32<true, false>(x, f_in, w_comb, f_in, weightings, hab, n, hab, f_in, 1, b_comb, sigmoid, 0, st);
}

size_t project_bwd_simt_workspace(int n, int f_in, int bd, int hab) {
  const size_t slabs = splitk_slabs(n);
  const size_t part = slabs * static_cast<size_t>(f_in) * std::max(bd, hab) * sizeof(float);
  return align_up(part, 256) + align_up(colsum_workspace_bytes(n, hab), 256) + 256;
}

int project_bwd_simt(const float* x, const float* w_bases, const float* w_comb, const float* d_bases,
                     const float* d_lin, int n, int f_in, int bd, int hab, float* d_x, float* d_w_bases,
                     float* d_w_comb, float* d_b_comb, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  EGC_REQUIRE(workspace_bytes >= project_bwd_simt_workspace(n, f_in, bd, hab), "egc_project_bwd: workspace too small");
  const int slabs = splitk_slabs(n);
  float* part = static_cast<float*>(workspace);
  void* colsum_ws = static_cast<char*>(workspace) +
                    align_up(static_cast<size_t>(slabs) * f_in * std::max(bd, hab) * sizeof(float), 256);
  if (d_x != nullptr) {
    // d_x[n,f_in] = d_bases[n,bd] . W_b[f_in,bd]^T  +  d_lin[n,hab] . W_c[hab,f_in]
    if (int rc = gemm_f32<true, false>(d_bases, bd, w_bases, bd, d_x, f_in, n, f_in, bd, 1, nullptr, 0, 0, st)) return rc;
    if (int rc = gemm_f32<true, true>(d_lin, hab, w_comb, f_in, d_x, f_in, n, f_in, hab, 1, nullptr, 0, 1, st)) return rc;
  }
  if (d_w_bases != nullptr) {
    // dW_b[f_in,bd] = x^T . d_bases  (split over node slabs, deterministic two-stage reduction)
    if (int rc = gemm_f32<false, true>(x, f_in, d_bases, bd, part, bd, f_in, bd, n, slabs, nullptr, 0, 0, st)) return rc;
    const int64_t count = static_cast<int64_t>(f_in) * bd;
    {
      LaunchScope egc_ls_("k_reduce_splits", st);
      k_reduce_splits<<<ceil_div(count, 256), 256, 0, st>>>(part, slabs, count, d_w_bases);
    }
    EGC_LAUNCH_CHECK("k_reduce_splits");
  }
  if (d_w_comb != nullptr) {
    // dW_c[hab,f_in] = d_lin^T . x
    if (int rc = gemm_f32<false, true>(d_lin, hab, x, f_in, part, f_in, hab, f_in, n, slabs, nullptr, 0, 0, st)) return rc;
    const int64_t count = static_cast<int64_t>(hab) * f_in;
    {
      LaunchScope egc_ls_("k_reduce_splits", st);
      k_reduce_splits<<<ceil_div(count, 256), 256, 0, st>>>(part, slabs, count, d_w_comb);
    }
    EGC_LAUNCH_CHECK("k_reduce_splits");
  }
  if (d_b_comb != nullptr) {
    if (int rc = colsum_f32(d_lin, n, hab, d_b_comb, colsum_ws, colsum_workspace_bytes(n, hab), st)) return rc;
  }
  return EGC_OK;
}

}  // namespace egc

using namespace egc;

extern "C" {

int egc_project_fwd(const float* x, const float* w_bases, const float* w_comb, const float* b_comb, int32_t n,
                    int32_t f_in, int32_t bd, int32_t hab, int32_t sigmoid, float* bases, float* weightings,
                    int32_t algo, void* stream) {
  EGC_REQUIRE(n > 0 && f_in > 0 && bd > 0 && hab > 0, "egc_project_fwd: n=%d f_in=%d bd=%d hab=%d", n, f_in, bd, hab);
  EGC_REQUIRE(x && w_bases && w_comb && bases && weightings, "egc_project_fwd: null pointer");
  EGC_REQUIRE(algo >= EGC_GEMM_AUTO && algo <= EGC_GEMM_TF32, "egc_project_fwd: unknown algo %d", algo);
  cudaStream_t st = as_stream(stream);
  const bool tc = algo != EGC_GEMM_FP32_SIMT && project_tc_supported(n, f_in, bd, hab);
  if (tc && tc_aligned(x, bases, weightings, b_comb)) {
    return project_fwd_tc(x, w_bases, w_comb, b_comb, n, f_in, bd, hab, sigmoid, bases, weightings,
                          algo == EGC_GEMM_TF32 ? 1 : 3, st);
  }
  if (algo == EGC_GEMM_3XTF32 || algo == EGC_GEMM_TF32) {
    if (tc) set_error("egc_project_fwd: tensor-core path does not support tensors that are not 16-byte aligned");
    else set_error("egc_project_fwd: tensor-core path does not support n=%d f_in=%d bd=%d hab=%d", n, f_in, bd, hab);
    return EGC_ERR_UNSUPPORTED;
  }
  return project_fwd_simt(x, w_bases, w_comb, b_comb, n, f_in, bd, hab, sigmoid, bases, weightings, st);
}

int egc_project_fwd_bf16(const float* x, const float* w_bases, const float* w_comb, const float* b_comb, int32_t n,
                         int32_t f_in, int32_t bd, int32_t hab, int32_t sigmoid, uint16_t* bases, float* weightings,
                         int32_t algo, void* stream) {
  EGC_REQUIRE(n > 0 && f_in > 0 && bd > 0 && hab > 0, "egc_project_fwd_bf16: n=%d f_in=%d bd=%d hab=%d", n, f_in, bd, hab);
  EGC_REQUIRE(x && w_bases && w_comb && bases && weightings, "egc_project_fwd_bf16: null pointer");
  EGC_REQUIRE(algo >= EGC_GEMM_AUTO && algo <= EGC_GEMM_TF32, "egc_project_fwd_bf16: unknown algo %d", algo);
  cudaStream_t st = as_stream(stream);
  const bool tc = algo != EGC_GEMM_FP32_SIMT && project_tc_supported(n, f_in, bd, hab);
  if (tc && tc_aligned(x, bases, weightings, b_comb)) {
    return project_fwd_tc_bf16(x, w_bases, w_comb, b_comb, n, f_in, bd, hab, sigmoid, bases, weightings,
                               algo == EGC_GEMM_TF32 ? 1 : 3, st);
  }
  if (algo == EGC_GEMM_3XTF32 || algo == EGC_GEMM_TF32) {
    if (tc) set_error("egc_project_fwd_bf16: tensor-core path does not support tensors that are not 16-byte aligned");
    else set_error("egc_project_fwd_bf16: tensor-core path does not support n=%d f_in=%d bd=%d hab=%d", n, f_in, bd, hab);
    return EGC_ERR_UNSUPPORTED;
  }
  return project_fwd_simt_bf16(x, w_bases, w_comb, b_comb, n, f_in, bd, hab, sigmoid, bases, weightings, st);
}

size_t egc_project_bwd_workspace_bytes(int32_t n, int32_t f_in, int32_t bd, int32_t hab) {
  if (n <= 0 || f_in <= 0 || bd <= 0 || hab <= 0) return 0;
  return std::max(project_bwd_simt_workspace(n, f_in, bd, hab), project_bwd_tc_workspace(n, f_in, bd, hab));
}

int egc_project_bwd(const float* x, const float* w_bases, const float* w_comb, const float* d_bases,
                    const float* d_lin, int32_t n, int32_t f_in, int32_t bd, int32_t hab, float* d_x,
                    float* d_w_bases, float* d_w_comb, float* d_b_comb, int32_t algo, void* workspace,
                    size_t workspace_bytes, void* stream) {
  EGC_REQUIRE(n > 0 && f_in > 0 && bd > 0 && hab > 0, "egc_project_bwd: n=%d f_in=%d bd=%d hab=%d", n, f_in, bd, hab);
  EGC_REQUIRE(x && w_bases && w_comb && d_bases && d_lin && workspace, "egc_project_bwd: null pointer");
  EGC_REQUIRE(algo >= EGC_GEMM_AUTO && algo <= EGC_GEMM_TF32, "egc_project_bwd: unknown algo %d", algo);
  cudaStream_t st = as_stream(stream);
  if (algo != EGC_GEMM_FP32_SIMT && project_tc_supported(n, f_in, bd, hab)) {
    if ((algo == EGC_GEMM_3XTF32 || algo == EGC_GEMM_TF32) && d_x != nullptr && !tc_aligned(d_bases, d_lin, d_x)) {
      set_error("egc_project_bwd: tensor-core path does not support tensors that are not 16-byte aligned");
      return EGC_ERR_UNSUPPORTED;
    }
    return project_bwd_tc(x, w_bases, w_comb, d_bases, d_lin, n, f_in, bd, hab, d_x, d_w_bases, d_w_comb, d_b_comb,
                          algo == EGC_GEMM_TF32 ? 1 : 3, workspace, workspace_bytes, st);
  }
  if (algo == EGC_GEMM_3XTF32 || algo == EGC_GEMM_TF32) {
    set_error("egc_project_bwd: tensor-core path does not support n=%d f_in=%d bd=%d hab=%d", n, f_in, bd, hab);
    return EGC_ERR_UNSUPPORTED;
  }
  return project_bwd_simt(x, w_bases, w_comb, d_bases, d_lin, n, f_in, bd, hab, d_x, d_w_bases, d_w_comb, d_b_comb,
                          workspace, workspace_bytes, st);
}

}  // extern "C"
