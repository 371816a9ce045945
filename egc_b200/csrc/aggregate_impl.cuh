// Kernel template of the fused forward aggregation + per-head combination.
// Included by aggregate_v{4,1}.cu, each of which instantiates one VEC family.
#pragma once

#include "aggregate.cuh"

namespace egc {

// ---------------------------------------------------------------------------------------------
// forward epilogue: out[row, h*D+d] = sum_ab w[h*AB+ab] * agg[ab*D+d] (+ bias)     (ref :195-208)
// agg rows live in this warp's shared memory as [A][BD] == [A*B][D].
// ---------------------------------------------------------------------------------------------
template <int EV, bool DROP = false>
__device__ __forceinline__ void combine_epilogue(const AggParams& p, const float* sm, int row, int lane) {
  const float* agg = sm + p.sm_agg;
  const float* w = sm + p.sm_w;
  float* out = p.out + static_cast<int64_t>(row) * p.HD;
  for (int o0 = lane * EV; o0 < p.HD; o0 += 32 * EV) {
    const int h = o0 / p.D, d = o0 - h * p.D;
    float acc[EV];
#pragma unroll
    for (int k = 0; k < EV; ++k) acc[k] = 0.f;
    const float* wh = w + h * p.AB;
    const float* ad = agg + d;
#pragma unroll 4
    for (int ab = 0; ab < p.AB; ++ab) {
      const float wv = wh[ab];
      float a[EV];
      ld_plain<EV>(a, ad + ab * p.D);
#pragma unroll
      for (int k = 0; k < EV; ++k) acc[k] = fmaf(wv, a[k], acc[k]);
    }
    if (p.bias != nullptr) {
#pragma unroll
      for (int k = 0; k < EV; ++k) acc[k] += __ldg(p.bias + o0 + k);
    }
#pragma unroll
    for (int k = 0; k < EV; ++k) {                            // BatchNorm-eval affine -> ReLU -> post-activation add
      if (p.epi_scale != nullptr) acc[k] = fmaf(acc[k], __ldg(p.epi_scale + o0 + k), __ldg(p.epi_shift + o0 + k));
      if (p.relu) acc[k] = fmaxf(acc[k], 0.f);
      if constexpr (!DROP) { if (p.epi_add != nullptr) acc[k] += p.epi_add[static_cast<int64_t>(row) * p.HD + o0 + k]; }
    }
    if constexpr (DROP) {                                     // ReLU -> dropout (one Philox draw per 4 columns) -> add
      if constexpr (EV == 4) dropout4(p, acc, row, o0);
      else acc[0] = dropout1(p, acc[0], row, o0);
      if (p.epi_add != nullptr) {
#pragma unroll
        for (int k = 0; k < EV; ++k) acc[k] += p.epi_add[static_cast<int64_t>(row) * p.HD + o0 + k];
      }
    }
    st_stream<EV>(out + o0, acc);
  }
}

// ---------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------
template <int MASK, int VEC, bool LINW, bool ARG, bool DROP = false>
__global__ void __launch_bounds__(kAggThreads, 3) k_aggregate(const __grid_constant__ AggParams p) {
  extern __shared__ __align__(16) float smem_all[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int gw = blockIdx.x * kAggWarps + warp;
  float* sm = smem_all + warp * p.sm_per_warp;

  int row, begin, end, chunk_id = -1, long_idx = -1;
  if (p.mode == 0) {
    if (gw < p.n_chunks) {
      chunk_id = gw;
      row = p.chunk_row[gw];
      begin = p.chunk_begin[gw];
      end = min(begin + EGC_CHUNK_EDGES, p.rowptr[row + 1]);
    } else {
      const int idx = gw - p.n_chunks;
      if (idx >= p.n_row_tasks) return;
      row = p.row_map != nullptr ? p.row_map[idx] : idx;
      begin = p.rowptr[row];
      end = p.rowptr[row + 1];
      if (end - begin > EGC_CHUNK_EDGES) return;      // long row: chunks + merge task do it
    }
  } else {
    long_idx = gw;
    if (long_idx >= p.n_long) return;
    row = p.long_rows[long_idx];
    begin = p.rowptr[row];
    end = p.rowptr[row + 1];
  }
  const bool is_chunk = chunk_id >= 0;
  const bool nonempty = end > begin;
  const float cntf = static_cast<float>(max(end - begin, 1));   // mean divides by the nnz count, min 1

  if (!is_chunk && p.out != nullptr) {   // stage this row's combination weights asynchronously
    const float* wsrc = p.weightings + static_cast<int64_t>(row) * p.HAB;
    for (int t = lane; t < p.HAB; t += 32) cp_async_4(sm + p.sm_w + t, wsrc + t);
  }

  const int G = p.G;
  for (int pass = 0; pass < p.n_pass; ++pass) {
    const int piece = pass * 32 + (lane & (G - 1));
    const bool active = piece < p.nvec;
    const int foff = min(piece, p.nvec - 1) * VEC;    // inactive lanes shadow the last piece, never write
    Acc<MASK, VEC, LINW, ARG> acc;
    acc.init();
    if (p.mode == 0) {
      accumulate_range<MASK, VEC, LINW, ARG>(acc, p, begin, end, lane, foff);
    } else {
      const int c0 = p.long_chunk_ptr[long_idx], c1 = p.long_chunk_ptr[long_idx + 1];
#pragma unroll 4
      for (int c = c0; c < c1; ++c)
        acc.merge_from(p.partials + (static_cast<int64_t>(c) * p.n_slots) * p.BD + foff, p.BD);
    }
    const bool writer = active && lane < G;    // after the xor merge every group holds the full result
    if (is_chunk) {
      if (writer) acc.store(p.partials + (static_cast<int64_t>(chunk_id) * p.n_slots) * p.BD + foff, p.BD);
      continue;
    }
    if (!writer) continue;
    float mean_slot[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) mean_slot[k] = 0.f;
    for (int a = 0; a < p.A; ++a) {
      const int code = p.aggr[a];
      float v[VEC], sv[VEC];
#pragma unroll
      for (int k = 0; k < VEC; ++k) {
        float mean = 0.f, var = 0.f;
        v[k] = finalize_one<MASK, VEC, LINW, ARG>(acc, code, k, cntf, nonempty, mean, var);
        sv[k] = v[k];
        if constexpr ((MASK & P_SQ) != 0) {
          if (code == EGC_AGGR_VAR || code == EGC_AGGR_STD) mean_slot[k] = mean;
          if (code == EGC_AGGR_STD && !(var > 0.f)) sv[k] = -v[k];   // sign bit = relu gate closed (std > 0 always)
        }
      }
      if (p.agg_init != nullptr) {                  // continue the sums of an earlier call (host: sum / symnorm only)
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
          v[k] += p.agg_init[(static_cast<int64_t>(row) * p.A + a) * p.BD + foff + k];
          sv[k] = v[k];
        }
      }
      if (p.out != nullptr) st_row<VEC>(sm + p.sm_agg + a * p.BD + foff, v);
      if (p.agg_out != nullptr) st_stream<VEC>(p.agg_out + (static_cast<int64_t>(row) * p.A + a) * p.BD + foff, v);
      if (p.saved != nullptr) st_stream<VEC>(p.saved + (static_cast<int64_t>(row) * p.n_saved + a) * p.BD + foff, sv);
      if constexpr (ARG) {
        float t[VEC];
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
          int arg = -1;
          if constexpr ((MASK & P_MAX) != 0) { if (code == EGC_AGGR_MAX) arg = acc.amx[k]; }
          if constexpr ((MASK & P_MIN) != 0) { if (code == EGC_AGGR_MIN) arg = acc.amn[k]; }
          t[k] = __int_as_float(arg);
        }
        if (p.arg_out != nullptr)
          st_stream<VEC>(reinterpret_cast<float*>(p.arg_out) + (static_cast<int64_t>(row) * p.A + a) * p.BD + foff, t);
        if (p.saved_arg != nullptr && p.arg_slot[a] >= 0)
          st_stream<VEC>(reinterpret_cast<float*>(p.saved_arg) +
                             (static_cast<int64_t>(row) * p.n_arg + p.arg_slot[a]) * p.BD + foff, t);
      }
    }
    if constexpr ((MASK & P_SQ) != 0) {
      if (p.saved != nullptr && p.n_saved > p.A)
        st_stream<VEC>(p.saved + (static_cast<int64_t>(row) * p.n_saved + p.A) * p.BD + foff, mean_slot);
    }
  }
  if (is_chunk || p.out == nullptr) return;

  cp_async_wait_all();
  __syncwarp();
  if (p.D % 4 == 0) combine_epilogue<4, DROP>(p, sm, row, lane);
  else combine_epilogue<1, DROP>(p, sm, row, lane);
}

// ---------------------------------------------------------------------------------------------
// dispatch over the primitive mask
// ---------------------------------------------------------------------------------------------
template <int MASK, int VEC, bool LINW, bool ARG, bool DROP = false>
int launch_one(const AggParams& p, int smem_bytes, cudaStream_t st) {
  auto kern = k_aggregate<MASK, VEC, LINW, ARG, DROP>;
  if (smem_bytes > 48 * 1024) {
    EGC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  }
  const int64_t tasks = p.mode == 0 ? static_cast<int64_t>(p.n_chunks) + p.n_row_tasks : p.n_long;
  if (tasks <= 0) return EGC_OK;
  const int grid = ceil_div(tasks, kAggWarps);
  {
    LaunchScope egc_ls_(p.mode ? "k_aggregate_fwd_merge" : "k_aggregate_fwd", st);
    kern<<<grid, kAggThreads, smem_bytes, st>>>(p);
  }
  EGC_LAUNCH_CHECK("k_aggregate");
  return EGC_OK;
}

// valid masks: any non-empty subset of {SUM, SYM, SQ, MAX, MIN} where SQ implies SUM
#define EGC_MASK_CASES(X) \
  X(1) X(2) X(3) X(5) X(7) X(8) X(9) X(10) X(11) X(13) X(15) X(16) X(17) X(18) X(19) X(21) X(23) \
  X(24) X(25) X(26) X(27) X(29) X(31)
// masks without SYM: the only ones that can carry per-nnz linear weights
#define EGC_MASK_CASES_NOSYM(X) X(1) X(5) X(8) X(9) X(13) X(16) X(17) X(21) X(24) X(25) X(29)

template <int MASK, int VEC, bool LINW, bool DROP = false>
int launch_arg(const AggParams& p, bool arg, int smem_bytes, cudaStream_t st) {
  if constexpr ((MASK & (P_MAX | P_MIN)) != 0) {
    if (arg) return launch_one<MASK, VEC, LINW, true, DROP>(p, smem_bytes, st);
  }
  return launch_one<MASK, VEC, LINW, false, DROP>(p, smem_bytes, st);
}

template <int VEC, bool DROP = false>
int launch_family(const AggParams& p, int mask, bool linw, bool arg, int smem_bytes, cudaStream_t st) {
  if (!linw) {
    switch (mask) {
#define X(M) case M: return launch_arg<M, VEC, false, DROP>(p, arg, smem_bytes, st);
      EGC_MASK_CASES(X)
#undef X
    }
  } else {
    switch (mask) {
#define X(M) case M: return launch_arg<M, VEC, true, DROP>(p, arg, smem_bytes, st);
      EGC_MASK_CASES_NOSYM(X)
#undef X
    }
  }
  set_error("aggregate: unsupported primitive mask %d (linw=%d)", mask, static_cast<int>(linw));
  return EGC_ERR_UNSUPPORTED;
}

}  // namespace egc
