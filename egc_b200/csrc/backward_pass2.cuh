// Backward pass 2 of the fused aggregation: per source column (CSC) gathers of the target-side streams, atomic-free.
// Column-block kernel (default) and the general warp-per-column kernel.  Included by aggregate_api.cu only.
#pragma once

#include "aggregate_fast.cuh"
#include "bf16.cuh"

namespace egc {

// =============================================================================================
// backward pass 2: per source column (CSC), gather of the target-side streams, atomic-free
// =============================================================================================
struct ScatterParams {
  const int32_t* colptr;
  const int32_t* rowidx;
  const float* val_sym;     // CSC order
  const float* val_lin;     // CSC order
  int n_cols;
  int col_begin, col_end;   // this launch covers source columns [col_begin, col_end) (and the long columns among them)
  int cols_per_task;        // column-block kernel: consecutive columns per task (<= kColsPerTask); fewer for small launches
  int n_long, n_chunks;
  const int32_t* long_rows;
  const int32_t* long_chunk_ptr;
  const int32_t* chunk_row;
  const int32_t* chunk_begin;
  float* partials;          // [n_chunks][n_ts][BD]
  const float* tstreams;    // [n_dst, n_ts, BD]
  const float* bases;       // [n_cols, BD]
  float* d_bases;           // [n_cols, BD]
  int n_ts, ts_sym, ts_lin, ts_sq;
  int64_t ts_row_stride;    // floats between the t-streams of consecutive target rows
  int64_t off_sym, off_lin, off_sq;   // float offset of each stream inside a target's row of interleaved streams
  int BD, nvec, G, n_pass;
  int routed;               // d_bases already holds a partial result (routed min/max gradients, earlier sweeps): accumulate
  int near_rows;            // column-block kernel: a gathered target row within this many rows of the column id is fetched
                            // with an L2 evict_last hint, the others evict_first (0: no hints).  Neighbouring columns of a
                            // locality-ordered graph gather the same near-diagonal rows again; far rows are one-off.
  int mode;
  int* long_counter;        // [n_long] zero on entry, or null: long columns are merged by a second launch (mode 1)
};

constexpr int kScatterUnroll = 4;

// single-stream instances are lean enough for 4 resident CTAs (<= 64 registers); multi-stream ones get 3
template <int TSMASK, int VEC, bool LINW>
__global__ void __launch_bounds__(kAggThreads, (TSMASK & (TSMASK - 1)) == 0 ? 4 : 3) k_scatter_bwd(const __grid_constant__ ScatterParams p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int gw = blockIdx.x * kAggWarps + warp;
  int colj, begin, end, chunk_id = -1, long_idx = -1;
  if (p.mode == 0) {
    if (gw < p.n_chunks) {
      chunk_id = gw;
      colj = p.chunk_row[gw];
      if (colj < p.col_begin || colj >= p.col_end) return;
      begin = p.chunk_begin[gw];
      end = min(begin + EGC_CHUNK_EDGES, p.colptr[colj + 1]);
    } else {
      colj = p.col_begin + (gw - p.n_chunks);
      if (colj >= p.col_end) return;
      begin = p.colptr[colj];
      end = p.colptr[colj + 1];
      if (end - begin > EGC_CHUNK_EDGES) return;
    }
  } else {
    long_idx = gw;
    if (long_idx >= p.n_long) return;
    colj = p.long_rows[long_idx];
    if (colj < p.col_begin || colj >= p.col_end) return;
    begin = p.colptr[colj];
    end = p.colptr[colj + 1];
  }
  const int G = p.G, NG = 32 / G, g = lane / G;
  const uint32_t row_stride = static_cast<uint32_t>(p.ts_row_stride);   // n_dst * row_stride < 2^32 (checked by the host)
  const int64_t part_stride = static_cast<int64_t>(p.n_ts) * p.BD;   // chunk partials stay interleaved

  for (int pass = 0; pass < p.n_pass; ++pass) {
    const int piece = pass * 32 + (lane & (G - 1));
    const bool active = piece < p.nvec;
    const int foff = min(piece, p.nvec - 1) * VEC;
    float a_sym[VEC], a_lin[VEC], a_sq[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) { a_sym[k] = 0.f; a_lin[k] = 0.f; a_sq[k] = 0.f; }

    if (p.mode == 0) {
      const float* __restrict__ src_sym = p.tstreams + p.off_sym + foff;
      const float* __restrict__ src_lin = p.tstreams + p.off_lin + foff;
      const float* __restrict__ src_sq = p.tstreams + p.off_sq + foff;
      const int last = end - 1;
      for (int e0 = begin + g; e0 < end + g; e0 += kScatterUnroll * NG) {
        int i[kScatterUnroll];
        float m[kScatterUnroll], vs[kScatterUnroll];
#pragma unroll
        for (int u = 0; u < kScatterUnroll; ++u) {
          const int e = e0 + u * NG, ec = min(e, last);
          i[u] = __ldg(p.rowidx + ec);
          m[u] = e <= last ? 1.f : 0.f;
          if constexpr (LINW) m[u] *= __ldg(p.val_lin + ec);
          vs[u] = 0.f;
          if constexpr ((TSMASK & 1) != 0) vs[u] = e <= last ? __ldg(p.val_sym + ec) : 0.f;
        }
        float xs[kScatterUnroll][VEC], xl[kScatterUnroll][VEC], xq[kScatterUnroll][VEC];
#pragma unroll
        for (int u = 0; u < kScatterUnroll; ++u) {
          const size_t r = static_cast<size_t>(static_cast<uint32_t>(i[u]) * row_stride);
          if constexpr ((TSMASK & 1) != 0) ld_row<VEC>(xs[u], src_sym + r);
          if constexpr ((TSMASK & 2) != 0) ld_row<VEC>(xl[u], src_lin + r);
          if constexpr ((TSMASK & 4) != 0) ld_row<VEC>(xq[u], src_sq + r);
        }
#pragma unroll
        for (int u = 0; u < kScatterUnroll; ++u) {
#pragma unroll
          for (int k = 0; k < VEC; ++k) {
            if constexpr ((TSMASK & 1) != 0) a_sym[k] = __fadd_rn(a_sym[k], __fmul_rn(xs[u][k], vs[u]));
            if constexpr ((TSMASK & 2) != 0) a_lin[k] = fmaf(xl[u][k], m[u], a_lin[k]);
            if constexpr ((TSMASK & 4) != 0) a_sq[k] = fmaf(xq[u][k], m[u], a_sq[k]);
          }
        }
      }
      for (int off = G; off < 32; off <<= 1) {
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
          if constexpr ((TSMASK & 1) != 0) a_sym[k] += __shfl_xor_sync(kFull, a_sym[k], off);
          if constexpr ((TSMASK & 2) != 0) a_lin[k] += __shfl_xor_sync(kFull, a_lin[k], off);
          if constexpr ((TSMASK & 4) != 0) a_sq[k] += __shfl_xor_sync(kFull, a_sq[k], off);
        }
      }
    } else {
      const int c0 = p.long_chunk_ptr[long_idx], c1 = p.long_chunk_ptr[long_idx + 1];
#pragma unroll 4
      for (int c = c0; c < c1; ++c) {
        const float* q = p.partials + static_cast<int64_t>(c) * part_stride + foff;
        float t[VEC];
        if constexpr ((TSMASK & 1) != 0) {
          ld_plain<VEC>(t, q + p.ts_sym * p.BD);
#pragma unroll
          for (int k = 0; k < VEC; ++k) a_sym[k] += t[k];
        }
        if constexpr ((TSMASK & 2) != 0) {
          ld_plain<VEC>(t, q + p.ts_lin * p.BD);
#pragma unroll
          for (int k = 0; k < VEC; ++k) a_lin[k] += t[k];
        }
        if constexpr ((TSMASK & 4) != 0) {
          ld_plain<VEC>(t, q + p.ts_sq * p.BD);
#pragma unroll
          for (int k = 0; k < VEC; ++k) a_sq[k] += t[k];
        }
      }
    }

    const bool writer = active && lane < G;
    if (chunk_id >= 0) {
      if (writer) {
        float* q = p.partials + static_cast<int64_t>(chunk_id) * part_stride + foff;
        if constexpr ((TSMASK & 1) != 0) st_row<VEC>(q + p.ts_sym * p.BD, a_sym);
        if constexpr ((TSMASK & 2) != 0) st_row<VEC>(q + p.ts_lin * p.BD, a_lin);
        if constexpr ((TSMASK & 4) != 0) st_row<VEC>(q + p.ts_sq * p.BD, a_sq);
      }
      if (p.long_counter == nullptr) continue;               // separate merge launch (mode 1) sums the partials
      // single-pass rows: the last chunk warp of the column to arrive sums all partials in chunk order
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
#pragma unroll
      for (int k = 0; k < VEC; ++k) { a_sym[k] = 0.f; a_lin[k] = 0.f; a_sq[k] = 0.f; }
      for (int c = c0; c < c1; ++c) {
        const float* q = p.partials + static_cast<int64_t>(c) * part_stride + foff;
        float t[VEC];
        if constexpr ((TSMASK & 1) != 0) {
          ld_cg<VEC>(t, q + p.ts_sym * p.BD);
#pragma unroll
          for (int k = 0; k < VEC; ++k) a_sym[k] += t[k];
        }
        if constexpr ((TSMASK & 2) != 0) {
          ld_cg<VEC>(t, q + p.ts_lin * p.BD);
#pragma unroll
          for (int k = 0; k < VEC; ++k) a_lin[k] += t[k];
        }
        if constexpr ((TSMASK & 4) != 0) {
          ld_cg<VEC>(t, q + p.ts_sq * p.BD);
#pragma unroll
          for (int k = 0; k < VEC; ++k) a_sq[k] += t[k];
        }
      }
      chunk_id = -1;                                         // falls through to the final write of column colj
    }
    if (!writer) continue;
    float* dst = p.d_bases + static_cast<int64_t>(colj) * p.BD + foff;
    float r[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) r[k] = 0.f;
    if (p.routed) ld_plain<VEC>(r, dst);
    if constexpr ((TSMASK & 4) != 0) {
      float xj[VEC];
      ld_row<VEC>(xj, p.bases + static_cast<int64_t>(colj) * p.BD + foff);
#pragma unroll
      for (int k = 0; k < VEC; ++k) r[k] += 2.f * xj[k] * a_sq[k];
    }
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      if constexpr ((TSMASK & 1) != 0) r[k] += a_sym[k];
      if constexpr ((TSMASK & 2) != 0) r[k] += a_lin[k];
    }
    st_row<VEC>(dst, r);
  }
}

template <int TSMASK, int VEC, bool LINW>
static int launch_scatter_one(const ScatterParams& p, cudaStream_t st) {
  const int64_t tasks = p.mode == 0 ? static_cast<int64_t>(p.n_chunks) + (p.col_end - p.col_begin) : p.n_long;
  if (tasks <= 0) return EGC_OK;
  {
    LaunchScope egc_ls_(p.mode ? "k_scatter_bwd_merge" : "k_scatter_bwd", st);
    k_scatter_bwd<TSMASK, VEC, LINW><<<ceil_div(tasks, kAggWarps), kAggThreads, 0, st>>>(p);
  }
  EGC_LAUNCH_CHECK("k_scatter_bwd");
  return EGC_OK;
}

template <int VEC, bool LINW>
static int launch_scatter_mask(const ScatterParams& p, int tsmask, cudaStream_t st) {
  switch (tsmask) {
    case 1: return launch_scatter_one<1, VEC, LINW>(p, st);
    case 2: return launch_scatter_one<2, VEC, LINW>(p, st);
    case 3: return launch_scatter_one<3, VEC, LINW>(p, st);
    case 4: return launch_scatter_one<4, VEC, LINW>(p, st);
    case 5: return launch_scatter_one<5, VEC, LINW>(p, st);
    case 6: return launch_scatter_one<6, VEC, LINW>(p, st);
    case 7: return launch_scatter_one<7, VEC, LINW>(p, st);
  }
  set_error("scatter_bwd: bad stream mask %d", tsmask);
  return EGC_ERR_UNSUPPORTED;
}

// ---------------------------------------------------------------------------------------------
// backward pass 2, column-block variant (the CSC twin of k_aggregate_rows, aggregate_rows.cuh): a task is a block of
// kColsPerTask CONSECUTIVE source columns handed out by an atomic counter; the column pointers are one coalesced
// load, the block's target ids / symnorm weights are one contiguous range staged into the warp's shared memory with
// cp.async in windows of kColWindow entries.  The warp-per-column kernel paid colptr -> rowidx -> gather (three
// dependent global latencies) for every column of ~15 entries.  Chunks of long columns run first (strided), merged by
// the last chunk warp to arrive.  128-bit pieces, unweighted entries, one pass (BD <= 128).
// ---------------------------------------------------------------------------------------------
constexpr int kColsPerTask = 8;
constexpr int kColWindow = 384;
static_assert(kColWindow >= EGC_CHUNK_EDGES, "a normal column must fit the staging window");

// four stored stream values -> fp32, with an L2 eviction hint
template <class ST>
__device__ __forceinline__ float4 ldg4_hint(const ST* p, uint64_t pol) {
  if constexpr (kBf16<ST>) {
    uint2 v;
    asm volatile("ld.global.nc.L2::cache_hint.v2.u32 {%0, %1}, [%2], %3;" : "=r"(v.x), "=r"(v.y) : "l"(p), "l"(pol));
    return widen_bf16x4(v);
  } else {
    return ldg_f4_hint(p, pol);
  }
}

// ST = storage type of the target-side streams and of `bases` (bf16: p.tstreams / p.bases point at bf16 rows; a lane still
// owns 4 features and sums them in fp32 in the same order)
template <int TSMASK, int G, bool HINT = false, class ST = float>
__global__ void __launch_bounds__(kAggThreads, (TSMASK & (TSMASK - 1)) == 0 ? 4 : 3) k_scatter_cols(const __grid_constant__ ScatterParams p, int* __restrict__ task_counter) {
  __shared__ int s_idx_all[kAggWarps][kColWindow];
  __shared__ float s_val_all[kAggWarps][(TSMASK & 1) ? kColWindow : 1];
  // entries in flight per lane group: single-stream instances have the registers for 8
  constexpr int NG = 32 / G, U = (TSMASK & (TSMASK - 1)) == 0 ? 2 * kScatterUnroll : kScatterUnroll, STEP = U * NG;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int* s_idx = s_idx_all[warp];
  float* s_val = s_val_all[warp];
  const int g = lane / G, piece = lane & (G - 1);
  const bool writer = piece < p.nvec && lane < G;
  const int foff = min(piece, p.nvec - 1) * 4;
  const uint32_t row_stride = static_cast<uint32_t>(p.ts_row_stride);   // n_dst * row_stride < 2^32 (checked by the host)
  const int64_t part_stride = static_cast<int64_t>(p.n_ts) * p.BD;
  const ST* __restrict__ src_sym = reinterpret_cast<const ST*>(p.tstreams) + p.off_sym + foff;
  const ST* __restrict__ src_lin = reinterpret_cast<const ST*>(p.tstreams) + p.off_lin + foff;
  const ST* __restrict__ src_sq = reinterpret_cast<const ST*>(p.tstreams) + p.off_sq + foff;
  float a_sym[4], a_lin[4], a_sq[4];

  auto stage = [&](int wb, int we) {                           // entries [wb, we) -> shared memory (we - wb <= kColWindow)
    for (int i = lane; i < we - wb; i += 32) {
      cp_async_4(s_idx + i, p.rowidx + wb + i);
      if constexpr ((TSMASK & 1) != 0) cp_async_4(s_val + i, p.val_sym + wb + i);
    }
    cp_async_wait_all();
    __syncwarp();
  };
  // sums over the staged entries [b, e) of one column (window base wb), then the xor-merge of the lane groups
  const uint64_t pol_near = HINT ? l2_policy_keep() : 0, pol_far = HINT ? l2_policy_stream() : 0;
  auto accumulate = [&](int b, int e, int wb, int colj) {
#pragma unroll
    for (int k = 0; k < 4; ++k) { a_sym[k] = 0.f; a_lin[k] = 0.f; a_sq[k] = 0.f; }
    for (int pos = b; pos < e; pos += STEP) {
      float m[U], vs[U];
      float4 xs[U], xl[U], xq[U];
      if constexpr (HINT) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int q = pos + u * NG + g, qc = min(q, e - 1);
          const int ti = s_idx[qc - wb];
          const size_t r = static_cast<size_t>(static_cast<uint32_t>(ti) * row_stride);
          const uint64_t pol = abs(ti - colj) <= p.near_rows ? pol_near : pol_far;
          m[u] = q < e ? 1.f : 0.f;
          vs[u] = 0.f;
          if constexpr ((TSMASK & 1) != 0) { vs[u] = q < e ? s_val[qc - wb] : 0.f; xs[u] = ldg4_hint<ST>(src_sym + r, pol); }
          if constexpr ((TSMASK & 2) != 0) xl[u] = ldg4_hint<ST>(src_lin + r, pol);
          if constexpr ((TSMASK & 4) != 0) xq[u] = ldg4_hint<ST>(src_sq + r, pol);
        }
      } else {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int q = pos + u * NG + g, qc = min(q, e - 1);
        const size_t r = static_cast<size_t>(static_cast<uint32_t>(s_idx[qc - wb]) * row_stride);
        m[u] = q < e ? 1.f : 0.f;
        vs[u] = 0.f;
        if constexpr ((TSMASK & 1) != 0) { vs[u] = q < e ? s_val[qc - wb] : 0.f; xs[u] = ldg4<ST>(src_sym + r); }
        if constexpr ((TSMASK & 2) != 0) xl[u] = ldg4<ST>(src_lin + r);
        if constexpr ((TSMASK & 4) != 0) xq[u] = ldg4<ST>(src_sq + r);
      }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if constexpr ((TSMASK & 1) != 0) {
          a_sym[0] = __fadd_rn(a_sym[0], __fmul_rn(xs[u].x, vs[u])); a_sym[1] = __fadd_rn(a_sym[1], __fmul_rn(xs[u].y, vs[u]));
          a_sym[2] = __fadd_rn(a_sym[2], __fmul_rn(xs[u].z, vs[u])); a_sym[3] = __fadd_rn(a_sym[3], __fmul_rn(xs[u].w, vs[u]));
        }
        if constexpr ((TSMASK & 2) != 0) {
          a_lin[0] = fmaf(xl[u].x, m[u], a_lin[0]); a_lin[1] = fmaf(xl[u].y, m[u], a_lin[1]);
          a_lin[2] = fmaf(xl[u].z, m[u], a_lin[2]); a_lin[3] = fmaf(xl[u].w, m[u], a_lin[3]);
        }
        if constexpr ((TSMASK & 4) != 0) {
          a_sq[0] = fmaf(xq[u].x, m[u], a_sq[0]); a_sq[1] = fmaf(xq[u].y, m[u], a_sq[1]);
          a_sq[2] = fmaf(xq[u].z, m[u], a_sq[2]); a_sq[3] = fmaf(xq[u].w, m[u], a_sq[3]);
        }
      }
    }
#pragma unroll
    for (int off = G; off < 32; off <<= 1) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if constexpr ((TSMASK & 1) != 0) a_sym[k] += __shfl_xor_sync(kFull, a_sym[k], off);
        if constexpr ((TSMASK & 2) != 0) a_lin[k] += __shfl_xor_sync(kFull, a_lin[k], off);
        if constexpr ((TSMASK & 4) != 0) a_sq[k] += __shfl_xor_sync(kFull, a_sq[k], off);
      }
    }
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

  // =========================== phase 0: chunks of long columns (strided over the grid) ===========================
  {
    const int warps_total = gridDim.x * kAggWarps;
    for (int chunk_id = blockIdx.x * kAggWarps + warp; chunk_id < p.n_chunks; chunk_id += warps_total) {
      const int colj = __ldg(p.chunk_row + chunk_id);
      if (colj < p.col_begin || colj >= p.col_end) continue;    // a long column outside this launch's range (warp-uniform)
      const int begin = __ldg(p.chunk_begin + chunk_id);
      const int end = min(begin + EGC_CHUNK_EDGES, __ldg(p.colptr + colj + 1));
      stage(begin, end);
      accumulate(begin, end, begin, colj);
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
#pragma unroll
      for (int k = 0; k < 4; ++k) { a_sym[k] = 0.f; a_lin[k] = 0.f; a_sq[k] = 0.f; }
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
      for (int c = ci; c < ci + n_fit; ++c) {
        const int b = __shfl_sync(kFull, cp, c), e = __shfl_sync(kFull, cpn, c);
        accumulate(b, e, wb, c0 + c);
        write_col(c0 + c);
      }
      ci += n_fit;
    }
    task = __shfl_sync(kFull, next_task, 0);
  }
}

template <int G, class ST = float>
static int launch_scatter_cols(const ScatterParams& p_in, int tsmask, int* task_counter, cudaStream_t st) {
  ScatterParams p = p_in;
  const int resident = (tsmask & (tsmask - 1)) == 0 ? 4 : 3;     // CTAs per SM, as the launch bounds
  {   // fewer columns per task when the launch is small (see pick_rows_per_task, aggregate_rows.cuh)
    const int64_t warps = static_cast<int64_t>(sm_count()) * resident * kAggWarps;
    int cpt = kColsPerTask;
    while (cpt > 1 && static_cast<int64_t>(p.col_end - p.col_begin) < 3 * warps * cpt) cpt >>= 1;
    p.cols_per_task = cpt;
  }
  const int n_blocks = ceil_div(p.col_end - p.col_begin, p.cols_per_task);
  const int grid = std::max(1, std::min(ceil_div(std::max(n_blocks, p.n_chunks), kAggWarps), sm_count() * resident));
  {
    LaunchScope egc_ls_("k_scatter_bwd", st);
#define EGC_SCATTER_COLS_CASE(M)                                                                           \
      case M:                                                                                              \
        if (p.near_rows > 0) k_scatter_cols<M, G, true, ST><<<grid, kAggThreads, 0, st>>>(p, task_counter); \
        else k_scatter_cols<M, G, false, ST><<<grid, kAggThreads, 0, st>>>(p, task_counter);                \
        break;
    switch (tsmask) {
      EGC_SCATTER_COLS_CASE(1) EGC_SCATTER_COLS_CASE(2) EGC_SCATTER_COLS_CASE(3) EGC_SCATTER_COLS_CASE(4)
      EGC_SCATTER_COLS_CASE(5) EGC_SCATTER_COLS_CASE(6) EGC_SCATTER_COLS_CASE(7)
      default: set_error("scatter_cols: bad stream mask %d", tsmask); return EGC_ERR_UNSUPPORTED;
    }
#undef EGC_SCATTER_COLS_CASE
  }
  EGC_LAUNCH_CHECK("k_scatter_cols");
  return EGC_OK;
}

static int launch_scatter(const ScatterParams& p, int tsmask, bool vec4, bool linw, cudaStream_t st) {
  if (vec4) return linw ? launch_scatter_mask<4, true>(p, tsmask, st) : launch_scatter_mask<4, false>(p, tsmask, st);
  return linw ? launch_scatter_mask<1, true>(p, tsmask, st) : launch_scatter_mask<1, false>(p, tsmask, st);
}



}  // namespace egc
