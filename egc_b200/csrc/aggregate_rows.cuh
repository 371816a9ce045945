// Row-block forward aggregation + per-head combination (sm_100a): the successor of k_aggregate_fast, for whole-graph
// calls and for row subsets (interior / boundary rows of a partitioned graph).  Same task model for long rows (chunk tasks, last chunk warp merges), same arithmetic and
// the same bits; what changes is how a warp finds and feeds its rows:
//
//   * a task is a block of kRowsPerTask CONSECUTIVE rows handed out by an atomic counter: the row pointers of the
//     block are one coalesced load, and the block's nnz are one contiguous range of `col` / `val_sym`;
//   * that range (and the block's combination weights, also contiguous) is staged into the warp's shared memory
//     with cp.async in windows of kWindow nnz, so the per-row chain  rowptr -> col -> gather  of the warp-per-row
//     kernel (three dependent global latencies per row) is paid once per window;
//   * software pipelining across rows: the first gather batch of row r+1 is issued BEFORE row r is finalized and
//     combined, so the ~400-instruction row epilogue overlaps the gather latency of the next row.
//
// The profile that motivated it (profiles/r01d, arxiv shape): 42 % of the issue slots of k_aggregate_fast were spent
// waiting on the first use of gathered rows, 12 % on the row-pointer / column-index loads.
#pragma once

#include "aggregate_fast.cuh"
#include "bf16.cuh"

namespace egc {

#ifndef EGC_ROWS_PER_TASK
#define EGC_ROWS_PER_TASK 8
#endif
#ifndef EGC_ROWS_UNROLL
#define EGC_ROWS_UNROLL 6        // gathers in flight per lane: 6 x 3 CTAs measured best (4: 0.271 ms, 6: 0.257, 8 x 2 CTAs: 0.267; arxiv shape)
#endif
#ifndef EGC_ROWS_CTAS
#define EGC_ROWS_CTAS 3
#endif
constexpr int kRowsPerTask = EGC_ROWS_PER_TASK;
constexpr int kWindow = 384;              // nnz staged at a time; >= EGC_CHUNK_EDGES so that every normal row fits
static_assert(kWindow >= EGC_CHUNK_EDGES, "a normal row must fit the staging window");

struct RowsSmem {                          // per-warp layout in floats, from A * BD and HAB
  int w, col, val, per_warp;               // aggregate staging starts at 0
  __host__ __device__ RowsSmem(int abd, int hab) {
    w = (abd + 3) & ~3;
    col = w + ((kRowsPerTask * hab + 3) & ~3);
    val = col + kWindow;
    per_warp = val + kWindow;
  }
};

// One 16-byte gather per lane and neighbour: 4 fp32 or 8 bf16 basis values (ST = the storage type of `bases`; p.bases
// then points at bf16 rows and p.nvec counts 8-wide pieces).  Values are widened to fp32 before any arithmetic.
template <class ST>
struct RowPiece {
  using T = float4;
  static constexpr int V = 4;
  static __device__ __forceinline__ T load(const ST* p, uint64_t pol) { return ldg_f4_hint(p, pol); }
};
template <>
struct RowPiece<bf16> {
  using T = uint4;
  static constexpr int V = 8;
  static __device__ __forceinline__ T load(const bf16* p, uint64_t pol) {
    uint4 v;
    asm volatile("ld.global.nc.L2::cache_hint.v4.u32 {%0, %1, %2, %3}, [%4], %5;"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p), "l"(pol));
    return v;
  }
};

template <int MASK, bool ARG>
__device__ __forceinline__ void add_edge(Acc<MASK, 8, false, ARG>& acc, const uint4& xv, float vs, int e) {
  const float x[8] = {bf16_lo(xv.x), bf16_hi(xv.x), bf16_lo(xv.y), bf16_hi(xv.y),
                      bf16_lo(xv.z), bf16_hi(xv.z), bf16_lo(xv.w), bf16_hi(xv.w)};
#pragma unroll
  for (int k = 0; k < 8; ++k) {          // the operations of add_edge<4> (aggregate_fast.cuh), per feature
    if constexpr (MASK & P_SUM) acc.sum[k] = __fadd_rn(acc.sum[k], x[k]);
    if constexpr (MASK & P_SQ) acc.sq[k] = fmaf(x[k], x[k], acc.sq[k]);
    if constexpr (MASK & P_SYM) acc.sym[k] = __fadd_rn(acc.sym[k], __fmul_rn(x[k], vs));
    if constexpr (MASK & P_MAX) {
      if constexpr (ARG) { if (x[k] > acc.mx[k]) { acc.mx[k] = x[k]; acc.amx[k] = e; } }
      else acc.mx[k] = fmaxf(acc.mx[k], x[k]);
    }
    if constexpr (MASK & P_MIN) {
      if constexpr (ARG) { if (x[k] < acc.mn[k]) { acc.mn[k] = x[k]; acc.amn[k] = e; } }
      else acc.mn[k] = fminf(acc.mn[k], x[k]);
    }
  }
}

// bf16 geometry of a layer configuration: 8-wide pieces, G = lanes per basis row (8 or 16 for rows of 40..128 values)
template <class Cfg>
struct Bf16Cfg : Cfg {
  static constexpr int nvec = Cfg::BD / 8;
  static constexpr int G = nvec > 8 ? 16 : 8;
  static_assert(Cfg::BD % 8 == 0 && nvec <= 16, "Bf16Cfg: basis rows of at most 128 values, a multiple of 8");
};

template <class Cfg, bool ARG, class ST = float, bool DROP = false>
__global__ void __launch_bounds__(kAggThreads, EGC_ROWS_CTAS) k_aggregate_rows(const __grid_constant__ AggParams p, int* __restrict__ task_counter) {
  extern __shared__ __align__(16) float smem_all[];
  constexpr int MASK = Cfg::MASK, G = Cfg::G;
  using GC = Get<Cfg>;
  constexpr int NG = 32 / G;
  constexpr int U = EGC_ROWS_UNROLL;
  using PC = RowPiece<ST>;
  constexpr int V = PC::V;                                      // features per lane
  constexpr int STEP = U * NG;                                  // nnz consumed by one batch of the warp
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const RowsSmem lay(GC::A(p) * GC::BD(p), GC::HAB(p));
  float* sm = smem_all + warp * lay.per_warp;
  float* s_agg = sm;
  float* s_w = sm + lay.w;
  int* s_col = reinterpret_cast<int*>(sm + lay.col);
  float* s_val = sm + lay.val;
  const int g = lane / G, li = lane & (G - 1);
  const bool writer = li < GC::nvec(p) && lane < G;                  // lanes of group 0 that own a real piece
  const int foff = min(li, GC::nvec(p) - 1) * V;                     // idle lanes shadow the last piece, never write
  const ST* __restrict__ src = reinterpret_cast<const ST*>(p.bases) + foff;
  const uint32_t BD = static_cast<uint32_t>(GC::BD(p));
  const uint64_t pol_keep = l2_policy_keep(), pol_stream = l2_policy_stream();
  using AccT = Acc<MASK, V, false, ARG>;
  const bool stage_w = p.out != nullptr;

  // epilogue geometry of this lane: outputs o = lane * EV + 32 * EV * it  ->  (weight row, offset in the head)
  const int EV = (GC::D(p) & 3) == 0 ? 4 : 1;
  int epi_w[kFastMaxIter], epi_d[kFastMaxIter];
#pragma unroll
  for (int it = 0; it < kFastMaxIter; ++it) {
    const int o = lane * EV + 32 * EV * it;
    const int h = o / GC::D(p);
    epi_w[it] = h * GC::AB(p);
    epi_d[it] = o - h * GC::D(p);
  }

  // ---- all aggregators of one finished row from its primitives, saved state, per-head combination (ref :195-208).
  // `w` = this row's combination weights in shared memory (cp.async may still be in flight: waited here).
  auto finalize = [&](int row, int begin, int end, const AccT& acc, const float* w) {
    if (writer) {
      const bool nonempty = end > begin;
      const float cntf = static_cast<float>(max(end - begin, 1));   // mean divides by the nnz count, min 1
      const float inv = __frcp_rn(cntf);
      float mean[V], var[V];
#pragma unroll
      for (int k = 0; k < V; ++k) { mean[k] = 0.f; var[k] = 0.f; }
      if constexpr ((MASK & P_SUM) != 0) {
#pragma unroll
        for (int k = 0; k < V; ++k) mean[k] = div_by(acc.sum[k], cntf, inv);
      }
      if constexpr ((MASK & P_SQ) != 0) {
#pragma unroll
        for (int k = 0; k < V; ++k)      // mean_sq - mean * mean, ref :242 / :271
          var[k] = __fsub_rn(div_by(acc.sq[k], cntf, inv), __fmul_rn(mean[k], mean[k]));
      }
      const size_t row_s = static_cast<size_t>(row);
#pragma unroll
      for (int a = 0; a < GC::A(p); ++a) {
        const int code = GC::aggr(p, a);
        float v[V], sv[V];
        int arg[V];
#pragma unroll
        for (int k = 0; k < V; ++k) { v[k] = 0.f; arg[k] = -1; }
        bool gate_sign = false;
        switch (code) {
          case EGC_AGGR_SUM:
            if constexpr ((MASK & P_SUM) != 0) { for (int k = 0; k < V; ++k) v[k] = acc.sum[k]; }
            break;
          case EGC_AGGR_MEAN:
            if constexpr ((MASK & P_SUM) != 0) { for (int k = 0; k < V; ++k) v[k] = mean[k]; }
            break;
          case EGC_AGGR_SYMNORM:
            if constexpr ((MASK & P_SYM) != 0) { for (int k = 0; k < V; ++k) v[k] = acc.sym[k]; }
            break;
          case EGC_AGGR_MAX:
            if constexpr ((MASK & P_MAX) != 0) {
              for (int k = 0; k < V; ++k) { v[k] = nonempty ? acc.mx[k] : 0.f; if constexpr (ARG) arg[k] = acc.amx[k]; }
            }
            break;
          case EGC_AGGR_MIN:
            if constexpr ((MASK & P_MIN) != 0) {
              for (int k = 0; k < V; ++k) { v[k] = nonempty ? acc.mn[k] : 0.f; if constexpr (ARG) arg[k] = acc.amn[k]; }
            }
            break;
          case EGC_AGGR_VAR:
            if constexpr ((MASK & P_SQ) != 0) { for (int k = 0; k < V; ++k) v[k] = var[k]; }
            break;
          case EGC_AGGR_STD:
            if constexpr ((MASK & P_SQ) != 0) {       // sqrt(relu(var) + 1e-5), ref :244 / :273
              for (int k = 0; k < V; ++k) v[k] = sqrtf(__fadd_rn(fmaxf(var[k], 0.f), kStdEps));
              gate_sign = true;
            }
            break;
        }
#pragma unroll
        for (int k = 0; k < V; ++k) sv[k] = (gate_sign && !(var[k] > 0.f)) ? -v[k] : v[k];   // sign bit = relu gate closed
#pragma unroll
        for (int h = 0; h < V; h += 4) {                     // 4 features per 128-bit store
          const float(&v4)[4] = *reinterpret_cast<const float(*)[4]>(v + h);
          const float(&sv4)[4] = *reinterpret_cast<const float(*)[4]>(sv + h);
          if (p.out != nullptr) st_row<4>(s_agg + a * BD + foff + h, v4);
          if (p.agg_out != nullptr) stg_f4_hint(p.agg_out + (row_s * GC::A(p) + a) * BD + foff + h, v4, pol_stream);
          if (p.saved != nullptr) stg_f4_hint(p.saved + (row_s * GC::n_saved(p) + a) * BD + foff + h, sv4, pol_stream);
          if constexpr (ARG) {
            const float t[4] = {__int_as_float(arg[h]), __int_as_float(arg[h + 1]), __int_as_float(arg[h + 2]), __int_as_float(arg[h + 3])};
            if (p.arg_out != nullptr)
              stg_f4_hint(reinterpret_cast<float*>(p.arg_out) + (row_s * GC::A(p) + a) * BD + foff + h, t, pol_stream);
            if (p.saved_arg != nullptr && GC::arg_slot(p, a) >= 0)
              stg_f4_hint(reinterpret_cast<float*>(p.saved_arg) + (row_s * GC::n_arg(p) + GC::arg_slot(p, a)) * BD + foff + h, t, pol_stream);
          }
        }
      }
      if constexpr ((MASK & P_SQ) != 0) {
#pragma unroll
        for (int h = 0; h < V; h += 4) {
          const float(&m4)[4] = *reinterpret_cast<const float(*)[4]>(mean + h);
          if (p.saved != nullptr && GC::n_saved(p) > GC::A(p)) stg_f4_hint(p.saved + (row_s * GC::n_saved(p) + GC::A(p)) * BD + foff + h, m4, pol_stream);
        }
      }
    }
    if (p.out == nullptr) return;
    __syncwarp();
    float* out = p.out + static_cast<int64_t>(row) * GC::HD(p);
    const int D = GC::D(p), AB = GC::AB(p);
#pragma unroll
    for (int it = 0; it < kFastMaxIter; ++it) {
      const int o = lane * EV + 32 * EV * it;
      if (o < GC::HD(p)) {
        const float* wh = w + epi_w[it];
        const float* ad = s_agg + epi_d[it];
        if (EV == 4) {
          float r[4] = {0.f, 0.f, 0.f, 0.f};
          if ((AB & 3) == 0) {                                 // weights of one head: whole 128-bit pieces (same order of FMAs)
#pragma unroll 3
            for (int ab = 0; ab < AB; ab += 4) {
              const float4 wv4 = *reinterpret_cast<const float4*>(wh + ab);
              const float wv[4] = {wv4.x, wv4.y, wv4.z, wv4.w};
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const float4 a = *reinterpret_cast<const float4*>(ad + (ab + q) * D);
                r[0] = fmaf(wv[q], a.x, r[0]); r[1] = fmaf(wv[q], a.y, r[1]); r[2] = fmaf(wv[q], a.z, r[2]); r[3] = fmaf(wv[q], a.w, r[3]);
              }
            }
          } else {
#pragma unroll 12
            for (int ab = 0; ab < AB; ++ab) {
              const float wv = wh[ab];
              const float4 a = *reinterpret_cast<const float4*>(ad + ab * D);
              r[0] = fmaf(wv, a.x, r[0]); r[1] = fmaf(wv, a.y, r[1]); r[2] = fmaf(wv, a.z, r[2]); r[3] = fmaf(wv, a.w, r[3]);
            }
          }
          if (p.bias != nullptr) {
            const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + o));
            r[0] += b.x; r[1] += b.y; r[2] += b.z; r[3] += b.w;
          }
          epilogue_tail4<DROP>(p, r, row, o, GC::HD(p));
          stg_f4_hint(out + o, r, pol_stream);
        } else {
          float r = 0.f;
#pragma unroll 4
          for (int ab = 0; ab < AB; ++ab) r = fmaf(wh[ab], ad[ab * D], r);
          if (p.bias != nullptr) r += __ldg(p.bias + o);
          r = epilogue_tail1<DROP>(p, r, row, o, GC::HD(p));
          __stcs(out + o, r);
        }
      }
    }
    __syncwarp();                                              // the next row overwrites the aggregate staging area
  };

  // =========================== phase 0: chunks of long rows (strided over the grid) ===========================
  {
    const int warps_total = gridDim.x * kAggWarps;
    for (int task = blockIdx.x * kAggWarps + warp; task < p.n_chunks; task += warps_total) {
      const int row = __ldg(p.chunk_row + task);
      const int begin = __ldg(p.chunk_begin + task);
      const int end = min(begin + EGC_CHUNK_EDGES, __ldg(p.rowptr + row + 1));
      AccT acc;
      acc.init();
      for (int e0 = begin; e0 < end; e0 += 32) {
        const int cnt = min(32, end - e0);
        int my_col = 0;
        float my_vs = 0.f;
        if (lane < cnt) {
          my_col = __ldg(p.col + e0 + lane);
          if constexpr (MASK & P_SYM) my_vs = __ldg(p.val_sym + e0 + lane);
        }
        for (int u0 = 0; u0 < cnt; u0 += STEP) {
          typename PC::T x[U];
          float vs[U];
#pragma unroll
          for (int t = 0; t < U; ++t) {
            const int u = min(u0 + t * NG + g, cnt - 1);
            const uint32_t j = static_cast<uint32_t>(__shfl_sync(kFull, my_col, u));
            vs[t] = 0.f;
            if constexpr (MASK & P_SYM) vs[t] = __shfl_sync(kFull, my_vs, u);
            x[t] = PC::load(src + static_cast<size_t>(j * BD), pol_keep);
          }
#pragma unroll
          for (int t = 0; t < U; ++t) {
            const int u = u0 + t * NG + g;
            if (u < cnt) add_edge<MASK, ARG>(acc, x[t], vs[t], e0 + u);
          }
        }
      }
      if constexpr (NG > 1) {
#pragma unroll
        for (int off = G; off < 32; off <<= 1) acc.merge_xor(off);
      }
      // publish the partial; the LAST chunk warp of the row to arrive merges all of them in chunk order (same result
      // whichever warp it is) and goes on to finalize the row
      if (writer) acc.store(p.partials + (static_cast<int64_t>(task) * p.n_slots) * BD + foff, BD);
      __threadfence();
      __syncwarp();
      int lo = 0, hi = p.n_long;                               // long row of this chunk: last l with long_chunk_ptr[l] <= task
      while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(p.long_chunk_ptr + mid) <= task) lo = mid; else hi = mid;
      }
      const int c0 = __ldg(p.long_chunk_ptr + lo), c1 = __ldg(p.long_chunk_ptr + lo + 1);
      int last = 0;
      if (lane == 0) last = atomicAdd(p.long_counter + lo, 1) == c1 - c0 - 1 ? 1 : 0;
      last = __shfl_sync(kFull, last, 0);
      if (!last) continue;
      __threadfence();
      if (lane == 0) p.long_counter[lo] = 0;                   // ready for the next launch
      acc.init();
      for (int c = c0; c < c1; ++c) acc.merge_from(p.partials + (static_cast<int64_t>(c) * p.n_slots) * BD + foff, BD);
      if (stage_w) {
        const float* wsrc = p.weightings + static_cast<int64_t>(row) * GC::HAB(p);
        for (int t = lane; t < GC::HAB(p); t += 32) cp_async_4(s_w + t, wsrc + t);
        cp_async_wait_all();
      }
      finalize(row, __ldg(p.rowptr + row), __ldg(p.rowptr + row + 1), acc, s_w);
    }
  }

  // =========================== phase 1: blocks of rows (dynamic) ===========================
  // Whole-graph calls: a block is kRowsPerTask CONSECUTIVE rows (one contiguous nnz range).  Row-subset calls (the
  // interior / boundary rows of a partitioned graph): kRowsPerTask consecutive entries of row_map, each row's range
  // staged on its own.  Lane l < nrows holds row l of the block: its id, [rp, rpn) and its offset in the window.
  const bool subset = p.row_map != nullptr;
  const int rpt = p.rows_per_task;                               // <= kRowsPerTask (the staging areas are sized for it)
  const int n_blocks = (p.n_row_tasks + rpt - 1) / rpt;
  int task = 0;
  if (lane == 0) task = atomicAdd(task_counter, 1);
  task = __shfl_sync(kFull, task, 0);
  while (task < n_blocks) {
    const int r0 = task * rpt;
    const int nrows = min(rpt, p.n_row_tasks - r0);
    int row_id, rp, rpn;
    if (subset) {
      row_id = __ldg(p.row_map + r0 + min(lane, nrows - 1));
      rp = __ldg(p.rowptr + row_id);
      rpn = __ldg(p.rowptr + row_id + 1);
    } else {
      row_id = r0 + lane;
      rp = __ldg(p.rowptr + r0 + min(lane, nrows));            // lanes 0..nrows hold the block's row pointers
      rpn = __shfl_down_sync(kFull, rp, 1);
    }
    int next_task = 0;
    if (lane == 0) next_task = atomicAdd(task_counter, 1);      // consumed at the end of this task
    const unsigned long_mask = __ballot_sync(kFull, lane < nrows && rpn - rp > EGC_CHUNK_EDGES);
    int ri = 0;
    while (ri < nrows) {
      if ((long_mask >> ri) & 1u) { ++ri; continue; }           // long row: its chunk tasks did it
      const unsigned later_long = long_mask >> ri;
      const int limit = later_long != 0u ? ri + __ffs(later_long) - 1 : nrows;
      // window offsets = running sum of the row lengths from row ri on; rows fit while the sum stays inside the window
      const int len = (lane >= ri && lane < limit) ? rpn - rp : 0;
      int incl = len;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(kFull, incl, d);
        if (lane >= d) incl += v;
      }
      const int woff = incl - len;
      const unsigned fit = __ballot_sync(kFull, lane >= ri && lane < limit && incl <= kWindow);
      const int n_fit = __popc(fit);                            // >= 1: a normal row has at most EGC_CHUNK_EDGES nnz
      const int total = __shfl_sync(kFull, incl, ri + n_fit - 1);
      // ---- stage the window: column ids, symnorm weights, the rows' combination weights
      __syncwarp();                                             // every lane is done reading the previous window
      if (!subset) {
        const int wb = __shfl_sync(kFull, rp, ri);
        for (int i = lane; i < total; i += 32) {
          cp_async_4(s_col + i, p.col + wb + i);
          if constexpr (MASK & P_SYM) cp_async_4(s_val + i, p.val_sym + wb + i);
        }
        if (stage_w) {
          const float* wsrc = p.weightings + static_cast<int64_t>(r0 + ri) * GC::HAB(p);
          const int nw = n_fit * GC::HAB(p);
          for (int t = lane; t < nw; t += 32) cp_async_4(s_w + t, wsrc + t);
        }
      } else {
        for (int r = ri; r < ri + n_fit; ++r) {
          const int rb = __shfl_sync(kFull, rp, r), rl = __shfl_sync(kFull, len, r), ro = __shfl_sync(kFull, woff, r);
          for (int i = lane; i < rl; i += 32) {
            cp_async_4(s_col + ro + i, p.col + rb + i);
            if constexpr (MASK & P_SYM) cp_async_4(s_val + ro + i, p.val_sym + rb + i);
          }
          if (stage_w) {
            const float* wsrc = p.weightings + static_cast<int64_t>(__shfl_sync(kFull, row_id, r)) * GC::HAB(p);
            for (int t = lane; t < GC::HAB(p); t += 32) cp_async_4(s_w + (r - ri) * GC::HAB(p) + t, wsrc + t);
          }
        }
      }
      cp_async_wait_all();
      __syncwarp();

      // gathers of one batch: positions b + t * NG + g clamped to the row's last nnz; wofs maps nnz position -> window
      typename PC::T x[U];
      auto issue = [&](int b, int e, int wofs) {
#pragma unroll
        for (int t = 0; t < U; ++t) {
          const int pos = min(b + t * NG + g, e - 1);
          const uint32_t j = static_cast<uint32_t>(s_col[pos + wofs]);
          x[t] = PC::load(src + static_cast<size_t>(j * BD), pol_keep);
        }
      };
      int b = __shfl_sync(kFull, rp, ri), e = __shfl_sync(kFull, rpn, ri);
      int wofs = __shfl_sync(kFull, woff, ri) - b;
      if (b < e) issue(b, e, wofs);
      for (int r = ri; r < ri + n_fit; ++r) {
        AccT acc;
        acc.init();
        for (int pos = b; pos < e;) {                           // x holds the batch that starts at pos
          if (pos + STEP <= e) {
#pragma unroll
            for (int t = 0; t < U; ++t) {
              const int q = pos + t * NG + g;
              float vs = 0.f;
              if constexpr (MASK & P_SYM) vs = s_val[q + wofs];
              add_edge<MASK, ARG>(acc, x[t], vs, q);
            }
          } else {
#pragma unroll
            for (int t = 0; t < U; ++t) {
              const int q = pos + t * NG + g;
              if (q < e) {
                float vs = 0.f;
                if constexpr (MASK & P_SYM) vs = s_val[q + wofs];
                add_edge<MASK, ARG>(acc, x[t], vs, q);
              }
            }
          }
          pos += STEP;
          if (pos < e) issue(pos, e, wofs);
        }
        if constexpr (NG > 1) {
#pragma unroll
          for (int off = G; off < 32; off <<= 1) acc.merge_xor(off);
        }
        int nb = 0, ne = 0, nwofs = 0;
        if (r + 1 < ri + n_fit) {                               // next row's first batch flies over this row's epilogue
          nb = __shfl_sync(kFull, rp, r + 1);
          ne = __shfl_sync(kFull, rpn, r + 1);
          nwofs = __shfl_sync(kFull, woff, r + 1) - nb;
          if (nb < ne) issue(nb, ne, nwofs);
        }
        finalize(__shfl_sync(kFull, row_id, r), b, e, acc, s_w + (r - ri) * GC::HAB(p));
        b = nb;
        e = ne;
        wofs = nwofs;
      }
      ri += n_fit;
    }
    task = __shfl_sync(kFull, next_task, 0);
  }
}

// ---------------------------------------------------------------------------------------------
// dispatch
// ---------------------------------------------------------------------------------------------
inline int rows_smem_bytes(const AggParams& p) {
  return RowsSmem(p.A * p.BD, p.HAB).per_warp * kAggWarps * static_cast<int>(sizeof(float));
}

// Rows per task: kRowsPerTask when there is enough work for every resident warp to get several tasks; a launch over few
// rows (one rank of an 8-way partition: ~21 k rows against 3552 resident warps) takes fewer, otherwise the kernel lasts
// as long as ONE serial 8-row task while most warps idle.
inline int pick_rows_per_task(int n_row_tasks) {
  const int64_t warps = static_cast<int64_t>(sm_count()) * EGC_ROWS_CTAS * kAggWarps;
  int rpt = kRowsPerTask;
  while (rpt > 1 && static_cast<int64_t>(n_row_tasks) < 3 * warps * rpt) rpt >>= 1;
  return rpt;
}

template <class Cfg, bool ARG, class ST = float, bool DROP = false>
int launch_rows_one(const AggParams& p_in, int* task_counter, cudaStream_t st) {
  AggParams p = p_in;
  p.rows_per_task = pick_rows_per_task(p.n_row_tasks);
  auto kern = k_aggregate_rows<Cfg, ARG, ST, DROP>;
  const int smem_bytes = rows_smem_bytes(p);
  if (smem_bytes > 48 * 1024) {
    EGC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  }
  const int n_blocks = ceil_div(p.n_row_tasks, p.rows_per_task);
  const int64_t warps_wanted = std::max<int64_t>(n_blocks, p.n_chunks);
  const int grid = static_cast<int>(std::min<int64_t>(ceil_div(warps_wanted, kAggWarps), static_cast<int64_t>(sm_count()) * EGC_ROWS_CTAS));
  {
    LaunchScope egc_ls_("k_aggregate_fwd", st);
    kern<<<grid, kAggThreads, smem_bytes, st>>>(p, task_counter);
  }
  EGC_LAUNCH_CHECK("k_aggregate_rows");
  return EGC_OK;
}

template <class Cfg, class ST = float, bool DROP = false>
int launch_rows_arg(const AggParams& p, bool arg, int* task_counter, cudaStream_t st) {
  if constexpr ((Cfg::MASK & (P_MAX | P_MIN)) != 0) {
    if (arg) return launch_rows_one<Cfg, true, ST, DROP>(p, task_counter, st);
  }
  return launch_rows_one<Cfg, false, ST, DROP>(p, task_counter, st);
}

template <int G, class ST = float, bool DROP = false>
int launch_rows_family(const AggParams& p, int mask, bool arg, int* task_counter, cudaStream_t st) {
  switch (mask) {
#define X(M) case M: return launch_rows_arg<DynCfg<M, G>, ST, DROP>(p, arg, task_counter, st);
    EGC_FAST_MASK_CASES(X)
#undef X
  }
  set_error("aggregate: unsupported primitive mask %d", mask);
  return EGC_ERR_UNSUPPORTED;
}

}  // namespace egc
