// Backward pass 2, ring variant of the column-block kernel (backward_pass2.cuh::k_scatter_cols) for 128-float rows
// (G = 32: one CSC entry = one warp-wide 512-byte row per target-side stream) and layers with two or more streams.
//
// k_scatter_cols gathers into registers: 4 entries x L streams x 16 bytes per lane, issued as one batch, waited for as one
// batch - so the queue drains at every batch and at every column boundary (a column has ~15 entries: four batches, each
// paying the full latency of rows that miss L2 half of the time; ncu r02p: 76 % of the warp stalls wait on those loads,
// DRAM at 51 % and L2 at 50 % of their peaks).  Here the rows land in a per-warp shared-memory ring instead:
//   * every lane copies ITS 16-byte piece of each stream with cp.async (no destination registers are held while the row is
//     in flight) into slot (q mod R) of the ring, one commit group per entry;
//   * the warp runs R entries ahead of the one it consumes, ACROSS the columns of its block (and across the batches of
//     a column): consuming entry q = wait_group(R - 1), three LDS.128 of the lane's own pieces, the same fp32 operations
//     in the same order as k_scatter_cols, then the freed slot takes entry q + R;
//   * a lane only ever reads what it wrote itself: no barrier, no bank conflict (lane l owns bytes [16 l, 16 l + 16)).
// Task model, chunk partials of long columns, the ordered merge and the epilogue are those of k_scatter_cols.
// bf16 streams (ST = bf16): a lane's piece is 8 bytes (4 features, still one lane per 4 features), a stream row 256 bytes,
// so a slot holds half the bytes and the same shared memory holds twice the ring depth.
#pragma once

#include "backward_pass2.cuh"
#include "tc_common.cuh"

namespace egc {

__device__ __forceinline__ void cp_async_16_hint(uint32_t smem_dst, const void* gmem_src, uint64_t pol) {
  asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;\n" ::"r"(smem_dst), "l"(gmem_src), "l"(pol) : "memory");
}
__device__ __forceinline__ void cp_async_8_hint(uint32_t smem_dst, const void* gmem_src, uint64_t pol) {
  asm volatile("cp.async.ca.shared.global.L2::cache_hint [%0], [%1], 8, %2;\n" ::"r"(smem_dst), "l"(gmem_src), "l"(pol) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }
__device__ __forceinline__ uint64_t l2_policy_normal() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}

template <int TSMASK, int R, class ST = float>
struct RingLayout {
  static constexpr int NS = (TSMASK & 1) + ((TSMASK >> 1) & 1) + ((TSMASK >> 2) & 1);
  static constexpr int kPieceBytes = 4 * static_cast<int>(sizeof(ST));   // one lane's 4 features of one stream
  static constexpr int kRowBytes = 32 * kPieceBytes;
  static constexpr int kSlotBytes = NS * kRowBytes;
  static constexpr int kIdxBytes = kColWindow * 4;
  static constexpr int kValBytes = (TSMASK & 1) ? kColWindow * 4 : 0;
  static constexpr int kWarpBytes = kIdxBytes + kValBytes + R * kSlotBytes;
  static constexpr int kCtaBytes = kAggWarps * kWarpBytes;
};

template <int TSMASK, int R, class ST = float>
__global__ void __launch_bounds__(kAggThreads, 3) k_scatter_ring(const __grid_constant__ ScatterParams p, int* __restrict__ task_counter) {
  extern __shared__ __align__(16) unsigned char ring_smem[];
  using L = RingLayout<TSMASK, R, ST>;
  constexpr uint32_t RB = L::kRowBytes;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char* base = ring_smem + warp * L::kWarpBytes;
  int* s_idx = reinterpret_cast<int*>(base);
  float* s_val = reinterpret_cast<float*>(base + L::kIdxBytes);
  const uint32_t ring_lane = smem_u32(base + L::kIdxBytes + L::kValBytes) + static_cast<uint32_t>(lane) * L::kPieceBytes;
  const bool writer = lane < p.nvec;
  const int foff = min(lane, p.nvec - 1) * 4;                    // idle lanes shadow the last piece, never write
  const uint32_t row_stride = static_cast<uint32_t>(p.ts_row_stride);
  const int64_t part_stride = static_cast<int64_t>(p.n_ts) * p.BD;
  const ST* __restrict__ src_sym = reinterpret_cast<const ST*>(p.tstreams) + p.off_sym + foff;
  const ST* __restrict__ src_lin = reinterpret_cast<const ST*>(p.tstreams) + p.off_lin + foff;
  const ST* __restrict__ src_sq = reinterpret_cast<const ST*>(p.tstreams) + p.off_sq + foff;
  const bool hinted = p.near_rows > 0;
  const uint64_t pol_near = hinted ? l2_policy_keep() : l2_policy_normal();
  const uint64_t pol_far = hinted ? l2_policy_stream() : pol_near;
  float a_sym[4] = {0.f, 0.f, 0.f, 0.f}, a_lin[4] = {0.f, 0.f, 0.f, 0.f}, a_sq[4] = {0.f, 0.f, 0.f, 0.f};
  int slot_w = 0, slot_r = 0;                                    // ring slot of the next entry to issue / to consume

  auto stage = [&](int wb, int we) {                             // entries [wb, we) -> shared memory (no ring group pending)
    for (int i = lane; i < we - wb; i += 32) {
      cp_async_4(s_idx + i, p.rowidx + wb + i);
      if constexpr ((TSMASK & 1) != 0) cp_async_4(s_val + i, p.val_sym + wb + i);
    }
    cp_async_wait_all();
    __syncwarp();
  };
  // entry with target row ti -> ring slot slot_w, one commit group (an empty group past the end keeps the count uniform)
  auto issue = [&](bool real, int ti, int col_ref) {
    if (real) {
      const size_t r = static_cast<size_t>(static_cast<uint32_t>(ti) * row_stride);
      const uint64_t pol = abs(ti - col_ref) <= p.near_rows ? pol_near : pol_far;
      uint32_t dst = ring_lane + static_cast<uint32_t>(slot_w) * L::kSlotBytes;
      auto cp = [&](uint32_t d, const ST* s) {
        if constexpr (kBf16<ST>) cp_async_8_hint(d, s, pol); else cp_async_16_hint(d, s, pol);
      };
      if constexpr ((TSMASK & 1) != 0) { cp(dst, src_sym + r); dst += RB; }
      if constexpr ((TSMASK & 2) != 0) { cp(dst, src_lin + r); dst += RB; }
      if constexpr ((TSMASK & 4) != 0) { cp(dst, src_sq + r); }
      slot_w = slot_w + 1 == R ? 0 : slot_w + 1;
    }
    cp_async_commit();
  };
  // consume the oldest entry in flight (weight vs) into the column sums - the arithmetic of k_scatter_cols::accumulate
  auto consume = [&](float vs) {
    cp_async_wait_group<R - 1>();
    uint32_t src = ring_lane + static_cast<uint32_t>(slot_r) * L::kSlotBytes;
    auto lds = [](uint32_t a) -> float4 {
      if constexpr (kBf16<ST>) {
        uint2 w;
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(w.x), "=r"(w.y) : "r"(a));
        return widen_bf16x4(w);
      } else {
        return lds128(a);
      }
    };
    if constexpr ((TSMASK & 1) != 0) {
      const float4 x = lds(src); src += RB;
      a_sym[0] = __fadd_rn(a_sym[0], __fmul_rn(x.x, vs)); a_sym[1] = __fadd_rn(a_sym[1], __fmul_rn(x.y, vs));
      a_sym[2] = __fadd_rn(a_sym[2], __fmul_rn(x.z, vs)); a_sym[3] = __fadd_rn(a_sym[3], __fmul_rn(x.w, vs));
    }
    if constexpr ((TSMASK & 2) != 0) {
      const float4 x = lds(src); src += RB;
      a_lin[0] += x.x; a_lin[1] += x.y; a_lin[2] += x.z; a_lin[3] += x.w;
    }
    if constexpr ((TSMASK & 4) != 0) {
      const float4 x = lds(src);
      a_sq[0] += x.x; a_sq[1] += x.y; a_sq[2] += x.z; a_sq[3] += x.w;
    }
    slot_r = slot_r + 1 == R ? 0 : slot_r + 1;
  };
  auto zero_sums = [&]() {
#pragma unroll
    for (int k = 0; k < 4; ++k) { a_sym[k] = 0.f; a_lin[k] = 0.f; a_sq[k] = 0.f; }
  };
  auto write_col = [&](int colj) {
    if (!writer) return;
    float* dst = p.d_bases + static_cast<int64_t>(colj) * p.BD + foff;
    float r[4] = {0.f, 0.f, 0.f, 0.f};
    if (p.routed) ld_plain<4>(r, dst);
    if constexpr ((TSMASK & 4) != 0) {
      float xj[4];
      ldg4<ST>(xj, reinterpret_cast<const ST*>(p.bases) + static_cast<int64_t>(colj) * p.BD + foff);
#pragma unroll
      for (int k = 0; k < 4; ++k) r[k] += 2.f * xj[k] * a_sq[k];
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if constexpr ((TSMASK & 1) != 0) r[k] += a_sym[k];
      if constexpr ((TSMASK & 2) != 0) r[k] += a_lin[k];
    }
    st_row<4>(dst, r);
  };
  // entries [wb, we) are staged; fills the ring with the first R of them
  auto prologue = [&](int wb, int we, int col_ref) {
    slot_w = 0; slot_r = 0;
#pragma unroll
    for (int k = 0; k < R; ++k) {
      const bool real = wb + k < we;
      issue(real, real ? s_idx[k] : 0, col_ref);
    }
  };

  // =========================== phase 0: chunks of long columns (strided over the grid) ===========================
  {
    const int warps_total = gridDim.x * kAggWarps;
    for (int chunk_id = blockIdx.x * kAggWarps + warp; chunk_id < p.n_chunks; chunk_id += warps_total) {
      const int colj = __ldg(p.chunk_row + chunk_id);
      if (colj < p.col_begin || colj >= p.col_end) continue;    // a long column outside this launch's range (warp-uniform)
      const int begin = __ldg(p.chunk_begin + chunk_id);
      const int end = min(begin + EGC_CHUNK_EDGES, __ldg(p.colptr + colj + 1));
      __syncwarp();
      stage(begin, end);
      prologue(begin, end, colj);
      zero_sums();
      for (int q = begin; q < end; ++q) {
        float vs = 0.f;
        if constexpr ((TSMASK & 1) != 0) vs = s_val[q - begin];
        consume(vs);
        const int qn = q + R;
        issue(qn < end, qn < end ? s_idx[qn - begin] : 0, colj);
      }
      if (writer) {
        float* q = p.partials + static_cast<int64_t>(chunk_id) * part_stride + foff;
        if constexpr ((TSMASK & 1) != 0) st_row<4>(q + p.ts_sym * p.BD, a_sym);
        if constexpr ((TSMASK & 2) != 0) st_row<4>(q + p.ts_lin * p.BD, a_lin);
        if constexpr ((TSMASK & 4) != 0) st_row<4>(q + p.ts_sq * p.BD, a_sq);
      }
      // the last chunk warp of the column to arrive sums all partials in chunk order and writes the column
      __threadfence();
      __syncwarp();
      int lo = 0, hi = p.n_long;
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(p.long_chunk_ptr + mid) <= chunk_id) lo = mid; else hi = mid;
      }
      const int c0 = __ldg(p.long_chunk_ptr + lo), c1 = __ldg(p.long_chunk_ptr + lo + 1);
      int last = 0;
      if (lane == 0) last = atomicAdd(p.long_counter + lo, 1) == c1 - c0 - 1 ? 1 : 0;
      last = __shfl_sync(kFull, last, 0);
      if (!last) continue;
      __threadfence();
      if (lane == 0) p.long_counter[lo] = 0;
      zero_sums();
      for (int c = c0; c < c1; ++c) {
        const float* q = p.partials + static_cast<int64_t>(c) * part_stride + foff;
        float t[4];
        if constexpr ((TSMASK & 1) != 0) {
          ld_cg<4>(t, q + p.ts_sym * p.BD);
#pragma unroll
          for (int k = 0; k < 4; ++k) a_sym[k] += t[k];
        }
        if constexpr ((TSMASK & 2) != 0) {
          ld_cg<4>(t, q + p.ts_lin * p.BD);
#pragma unroll
          for (int k = 0; k < 4; ++k) a_lin[k] += t[k];
        }
        if constexpr ((TSMASK & 4) != 0) {
          ld_cg<4>(t, q + p.ts_sq * p.BD);
#pragma unroll
          for (int k = 0; k < 4; ++k) a_sq[k] += t[k];
        }
      }
      write_col(colj);
    }
  }

  // =========================== phase 1: blocks of consecutive columns (dynamic) ===========================
  const int cpt = p.cols_per_task;
  const int n_blocks = (p.col_end - p.col_begin + cpt - 1) / cpt;
  int task = 0;
  if (lane == 0) task = atomicAdd(task_counter, 1);
  task = __shfl_sync(kFull, task, 0);
  while (task < n_blocks) {
    const int c0 = p.col_begin + task * cpt;
    const int ncols = min(cpt, p.col_end - c0);
    const int cp = __ldg(p.colptr + c0 + min(lane, ncols));    // lanes 0..ncols hold the block's column pointers
    int next_task = 0;
    if (lane == 0) next_task = atomicAdd(task_counter, 1);      // consumed at the end of this task
    const int cpn = __shfl_down_sync(kFull, cp, 1);             // lane l < ncols: column l = [cp, cpn)
    const unsigned long_mask = __ballot_sync(kFull, lane < ncols && cpn - cp > EGC_CHUNK_EDGES);
    int ci = 0;
    while (ci < ncols) {
      if ((long_mask >> ci) & 1u) { ++ci; continue; }           // long column: its chunk tasks did it
      const unsigned later_long = long_mask >> ci;
      const int limit = later_long != 0u ? ci + __ffs(later_long) - 1 : ncols;
      const int wb = __shfl_sync(kFull, cp, ci);
      const unsigned fit = __ballot_sync(kFull, lane >= ci && lane < limit && cpn - wb <= kColWindow);
      const int n_fit = __popc(fit);                            // >= 1
      const int we = __shfl_sync(kFull, cpn, ci + n_fit - 1);
      __syncwarp();                                             // every lane is done with the previous window
      stage(wb, we);
      prologue(wb, we, c0);
      int qn = wb + R;                                          // next entry to issue: the ring runs ahead across columns
      for (int c = ci; c < ci + n_fit; ++c) {
        const int b = __shfl_sync(kFull, cp, c), e = __shfl_sync(kFull, cpn, c);
        zero_sums();
        for (int q = b; q < e; ++q, ++qn) {
          float vs = 0.f;
          if constexpr ((TSMASK & 1) != 0) vs = s_val[q - wb];
          consume(vs);
          issue(qn < we, qn < we ? s_idx[qn - wb] : 0, c0);
        }
        write_col(c0 + c);
      }
      ci += n_fit;
    }
    task = __shfl_sync(kFull, next_task, 0);
  }
}

// ring depth picked by the host: 4 (three CTAs per SM) or 7 (two CTAs per SM) for a three-stream fp32 layer
template <int R, class ST = float>
static int launch_scatter_ring(const ScatterParams& p_in, int tsmask, int* task_counter, cudaStream_t st) {
  ScatterParams p = p_in;
#define EGC_RING_CASE(M)                                                                                         \
  case M: {                                                                                                      \
    using L = RingLayout<M, R, ST>;                                                                              \
    const int resident = std::max(1, std::min(3, (227 * 1024) / (L::kCtaBytes + 1024)));                         \
    const int64_t warps = static_cast<int64_t>(sm_count()) * resident * kAggWarps;                               \
    int cpt = kColsPerTask;                                                                                      \
    while (cpt > 1 && static_cast<int64_t>(p.col_end - p.col_begin) < 3 * warps * cpt) cpt >>= 1;                \
    p.cols_per_task = cpt;                                                                                       \
    const int n_blocks = ceil_div(p.col_end - p.col_begin, p.cols_per_task);                                     \
    const int grid = std::max(1, std::min(ceil_div(std::max(n_blocks, p.n_chunks), kAggWarps), sm_count() * resident)); \
    auto kern = k_scatter_ring<M, R, ST>;                                                                        \
    EGC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kCtaBytes));             \
    LaunchScope egc_ls_("k_scatter_bwd", st);                                                                    \
    kern<<<grid, kAggThreads, L::kCtaBytes, st>>>(p, task_counter);                                              \
  } break;
  switch (tsmask) {
    EGC_RING_CASE(3) EGC_RING_CASE(5) EGC_RING_CASE(6) EGC_RING_CASE(7)
    default: set_error("scatter_ring: stream mask %d has fewer than two streams", tsmask); return EGC_ERR_UNSUPPORTED;
  }
#undef EGC_RING_CASE
  EGC_LAUNCH_CHECK("k_scatter_ring");
  return EGC_OK;
}

}  // namespace egc
