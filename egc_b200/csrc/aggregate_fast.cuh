// Fast path of the fused forward aggregation + per-head combination (sm_100a): basis rows of at most
// 128 floats (one 128-bit piece per lane), unweighted messages.  Same task model, partial layout and
// results as k_aggregate (aggregate_impl.cuh), which remains the general kernel (wide rows, scalar rows,
// per-nnz linear weights, long-row merges).
//
// What makes it fast:
//   * persistent warps: a grid of (SMs x resident CTAs) walks the task list with a stride, so the lane
//     geometry and the epilogue's (head, offset) decomposition are computed once, not per row;
//   * column indices / symnorm weights of 32 nnz are fetched with ONE coalesced load per lane and
//     broadcast with shuffles; the row gathers are issued kFastUnroll at a time before any arithmetic;
//   * the lane group size G is a template parameter: G = 32 -> one neighbour per step, G = 16 -> two;
//   * tails are handled with (group-)uniform predicates instead of padded slots;
//   * 32-bit index arithmetic everywhere except the final row address.
#pragma once

#include "aggregate.cuh"

namespace egc {

constexpr int kFastUnroll = 4;
constexpr int kFastMaxIter = 4;      // epilogue iterations (outputs per lane) whose (h, d) are kept in registers

// L2 eviction policies: gathered basis rows are re-read ~deg times (keep), everything else streams
__device__ __forceinline__ uint64_t l2_policy_keep() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint64_t l2_policy_stream() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ float4 ldg_f4_hint(const float* p, uint64_t pol) {
  float4 v;
  asm volatile("ld.global.nc.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ void stg_f4_hint(float* p, const float (&v)[4], uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;"
               ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "l"(pol) : "memory");
}

// tail of the output epilogue after bias: BatchNorm-eval affine -> ReLU -> [DROP: dropout] -> post-activation add
// (egc_epilogue order)
template <bool DROP = false>
__device__ __forceinline__ void epilogue_tail4(const AggParams& p, float (&r)[4], int64_t row, int o, int HD) {
  if (p.epi_scale != nullptr) {
    const float4 sc = __ldg(reinterpret_cast<const float4*>(p.epi_scale + o)), sh = __ldg(reinterpret_cast<const float4*>(p.epi_shift + o));
    r[0] = fmaf(r[0], sc.x, sh.x); r[1] = fmaf(r[1], sc.y, sh.y); r[2] = fmaf(r[2], sc.z, sh.z); r[3] = fmaf(r[3], sc.w, sh.w);
  }
  if (p.relu) { r[0] = fmaxf(r[0], 0.f); r[1] = fmaxf(r[1], 0.f); r[2] = fmaxf(r[2], 0.f); r[3] = fmaxf(r[3], 0.f); }
  if constexpr (DROP) dropout4(p, r, row, o);
  if (p.epi_add != nullptr) {
    const float4 a = *reinterpret_cast<const float4*>(p.epi_add + row * HD + o);
    r[0] += a.x; r[1] += a.y; r[2] += a.z; r[3] += a.w;
  }
}
template <bool DROP = false>
__device__ __forceinline__ float epilogue_tail1(const AggParams& p, float r, int64_t row, int o, int HD) {
  if (p.epi_scale != nullptr) r = fmaf(r, __ldg(p.epi_scale + o), __ldg(p.epi_shift + o));
  if (p.relu) r = fmaxf(r, 0.f);
  if constexpr (DROP) r = dropout1(p, r, row, o);
  if (p.epi_add != nullptr) r += p.epi_add[row * HD + o];
  return r;
}

// x / c with r = 1 / c (IEEE reciprocal): one Newton correction of the quotient (correctly rounded up to rare
// double-rounding cases; exact whenever the quotient is representable)
__device__ __forceinline__ float div_by(float x, float c, float r) {
  const float q = x * r;
  return fmaf(fmaf(-q, c, x), r, q);
}


// ---------------------------------------------------------------------------------------------
// Layer configurations.  DynCfg reads every dimension from the kernel parameters (any layer).  StaticCfg bakes
// heads / bases / head dim / the ordered aggregator list into the kernel: loops over aggregators, bases and
// heads unroll, the finalize switch folds, all index arithmetic becomes immediate.  Both produce the same bits.
// ---------------------------------------------------------------------------------------------
template <int MASK_, int G_>
struct DynCfg {
  static constexpr bool kStatic = false;
  static constexpr int MASK = MASK_, G = G_;
};

constexpr int cfg_a4(int v) { return (v + 3) & ~3; }

template <int H_, int B_, int D_, int... C>
struct StaticCfg {
  static constexpr bool kStatic = true;
  static constexpr int H = H_, B = B_, D = D_, A = sizeof...(C);
  static constexpr int BD = B * D, HD = H * D, AB = A * B, HAB = H * AB;
  static __host__ __device__ constexpr int code(int a) {
    constexpr int arr[] = {C...};
    return arr[a];
  }
  static constexpr int mask_of() {
    int m = 0;
    for (int a = 0; a < A; ++a) {
      const int c = code(a);
      if (c == EGC_AGGR_SUM || c == EGC_AGGR_MEAN) m |= P_SUM;
      if (c == EGC_AGGR_SYMNORM) m |= P_SYM;
      if (c == EGC_AGGR_MAX) m |= P_MAX;
      if (c == EGC_AGGR_MIN) m |= P_MIN;
      if (c == EGC_AGGR_VAR || c == EGC_AGGR_STD) m |= P_SUM | P_SQ;
    }
    return m;
  }
  static constexpr int MASK = mask_of();
  static constexpr int nvec = BD / 4;
  static constexpr int G = nvec > 16 ? 32 : 16;
  static constexpr bool has_var = (MASK & P_SQ) != 0;
  static constexpr int n_saved = A + (has_var ? 1 : 0);
  static __host__ __device__ constexpr int arg_slot(int a) {
    if (code(a) != EGC_AGGR_MAX && code(a) != EGC_AGGR_MIN) return -1;
    int n = 0;
    for (int i = 0; i < a; ++i) n += (code(i) == EGC_AGGR_MAX || code(i) == EGC_AGGR_MIN) ? 1 : 0;
    return n;
  }
  static constexpr int n_arg = ((MASK & P_MAX) ? 1 : 0) * 0 + []() constexpr { int n = 0; for (int a = 0; a < A; ++a) n += (code(a) == EGC_AGGR_MAX || code(a) == EGC_AGGR_MIN) ? 1 : 0; return n; }();
  static constexpr int sm_agg = 0, sm_w = cfg_a4(A * BD), sm_per_warp = cfg_a4(sm_w + HAB);
  // backward pass 1: per-warp staging layout and target-side stream slots (same rules as the host code)
  static constexpr int bsm_w = 0, bsm_g = cfg_a4(HAB), bsm_saved = cfg_a4(bsm_g + HD);
  static constexpr int bsm_arg = cfg_a4(bsm_saved + n_saved * BD), bsm_per_warp = cfg_a4(bsm_arg + n_arg * BD);
  static constexpr bool has_lin = (MASK & P_SUM) != 0;
  static constexpr int ts_sym = (MASK & P_SYM) ? 0 : -1;
  static constexpr int ts_lin = has_lin ? ((MASK & P_SYM) ? 1 : 0) : -1;
  static constexpr int ts_sq = has_var ? ((MASK & P_SYM) ? 1 : 0) + (has_lin ? 1 : 0) : -1;
  static_assert(BD % 4 == 0 && D % 4 == 0 && nvec > 8 && nvec <= 32, "StaticCfg: basis rows of 36..128 floats, D % 4 == 0");
  static bool matches(const egc_layer_desc& d) {
    if (d.heads != H || d.bases != B || d.dim != D || d.n_aggr != A) return false;
    for (int a = 0; a < A; ++a) if (d.aggr[a] != code(a)) return false;
    return true;
  }
};

// the specialised layer shapes (heads, bases, head dim, aggregators in constructor order).  BASELINE.json
// configs 2 / 3 / 5 are the first, config 4 the second; the others are the reference's EGC-S / EGC-M variants
// at hidden 128 (ref experiments/*/configs.py); 4 / 5 are REGConv's relation and root terms (ref rmag/models.py).
// Every other layer runs the DynCfg kernels.
#define EGC_STATIC_CFGS(X)                                               \
  X(0, 4, 4, 32, EGC_AGGR_SYMNORM, EGC_AGGR_MAX, EGC_AGGR_STD)           \
  X(1, 8, 4, 16, EGC_AGGR_SYMNORM)                                       \
  X(2, 4, 4, 32, EGC_AGGR_SYMNORM)                                       \
  X(3, 4, 4, 32, EGC_AGGR_SYMNORM, EGC_AGGR_MAX, EGC_AGGR_MEAN)          \
  X(4, 8, 4, 16, EGC_AGGR_MEAN, EGC_AGGR_MAX)                            \
  X(5, 8, 4, 16, EGC_AGGR_SUM)

inline int static_cfg_index(const egc_layer_desc& d) {
#define X(I, ...) if (StaticCfg<__VA_ARGS__>::matches(d)) return I;
  EGC_STATIC_CFGS(X)
#undef X
  return -1;
}

// same idea for the parameter block of backward pass 1 (CombineBwdParams, backward_pass1.cuh)
template <class Cfg, class P>
struct GetB {
#define EGC_GETB(name, sname)                                                                 \
  static __device__ __forceinline__ int name(const P& p) {                                    \
    if constexpr (Cfg::kStatic) return Cfg::sname; else return p.name;                         \
  }
  EGC_GETB(H, H) EGC_GETB(B, B) EGC_GETB(D, D) EGC_GETB(A, A) EGC_GETB(BD, BD) EGC_GETB(HD, HD) EGC_GETB(AB, AB)
  EGC_GETB(HAB, HAB) EGC_GETB(n_saved, n_saved) EGC_GETB(n_arg, n_arg) EGC_GETB(sm_w, bsm_w) EGC_GETB(sm_g, bsm_g)
  EGC_GETB(sm_saved, bsm_saved) EGC_GETB(sm_arg, bsm_arg) EGC_GETB(sm_per_warp, bsm_per_warp)
  EGC_GETB(ts_sym, ts_sym) EGC_GETB(ts_lin, ts_lin) EGC_GETB(ts_sq, ts_sq)
#undef EGC_GETB
  static __device__ __forceinline__ int aggr(const P& p, int a) {
    if constexpr (Cfg::kStatic) return Cfg::code(a); else return p.aggr[a];
  }
  static __device__ __forceinline__ int arg_slot(const P& p, int a) {
    if constexpr (Cfg::kStatic) return Cfg::arg_slot(a); else return p.arg_slot[a];
  }
};

template <class Cfg>
struct Get {
#define EGC_GET(name)                                                                         \
  static __device__ __forceinline__ int name(const AggParams& p) {                            \
    if constexpr (Cfg::kStatic) return Cfg::name; else return p.name;                          \
  }
  EGC_GET(H) EGC_GET(B) EGC_GET(D) EGC_GET(A) EGC_GET(BD) EGC_GET(HD) EGC_GET(AB) EGC_GET(HAB)
  EGC_GET(nvec) EGC_GET(n_saved) EGC_GET(n_arg) EGC_GET(sm_agg) EGC_GET(sm_w) EGC_GET(sm_per_warp)
#undef EGC_GET
  static __device__ __forceinline__ int aggr(const AggParams& p, int a) {
    if constexpr (Cfg::kStatic) return Cfg::code(a); else return p.aggr[a];
  }
  static __device__ __forceinline__ int arg_slot(const AggParams& p, int a) {
    if constexpr (Cfg::kStatic) return Cfg::arg_slot(a); else return p.arg_slot[a];
  }
};

template <int MASK, bool ARG>
__device__ __forceinline__ void add_edge(Acc<MASK, 4, false, ARG>& acc, const float4& xv, float vs, int e) {
  const float x[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if constexpr (MASK & P_SUM) acc.sum[k] = __fadd_rn(acc.sum[k], x[k]);
    if constexpr (MASK & P_SQ) acc.sq[k] = fmaf(x[k], x[k], acc.sq[k]);
    // separate multiply and add: a sequential walk reproduces the reference's fp32 symnorm sums bit for bit
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

template <class Cfg, bool ARG, bool DROP = false>
__global__ void __launch_bounds__(kAggThreads, 4) k_aggregate_fast(const __grid_constant__ AggParams p) {
  extern __shared__ __align__(16) float smem_all[];
  constexpr int MASK = Cfg::MASK, G = Cfg::G;
  using GC = Get<Cfg>;
  constexpr int NG = 32 / G;
  constexpr int STEP = kFastUnroll * NG;                        // nnz consumed by one batch of the warp
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* sm = smem_all + warp * GC::sm_per_warp(p);
  const int g = lane / G, li = lane & (G - 1);
  const bool writer = li < GC::nvec(p) && lane < G;                  // lanes of group 0 that own a real piece
  const int foff = min(li, GC::nvec(p) - 1) * 4;                     // idle lanes shadow the last piece, never write
  const float* __restrict__ src = p.bases + foff;
  const uint32_t BD = static_cast<uint32_t>(GC::BD(p));
  const int n_tasks = p.n_chunks + p.n_row_tasks;
  const int warps_total = gridDim.x * kAggWarps;
  const uint64_t pol_keep = l2_policy_keep(), pol_stream = l2_policy_stream();
  using AccT = Acc<MASK, 4, false, ARG>;

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

  for (int task = blockIdx.x * kAggWarps + warp; task < n_tasks; task += warps_total) {
    int row, begin, end;
    bool is_chunk = task < p.n_chunks;
    if (is_chunk) {
      row = __ldg(p.chunk_row + task);
      begin = __ldg(p.chunk_begin + task);
      end = min(begin + EGC_CHUNK_EDGES, __ldg(p.rowptr + row + 1));
    } else {
      const int idx = task - p.n_chunks;
      row = p.row_map != nullptr ? __ldg(p.row_map + idx) : idx;
      begin = __ldg(p.rowptr + row);
      end = __ldg(p.rowptr + row + 1);
      if (end - begin > EGC_CHUNK_EDGES) continue;            // long row: its chunk tasks do it
    }
    const bool stage_w = p.out != nullptr;
    if (!is_chunk && stage_w) {                                // stage this row's combination weights asynchronously
      const float* wsrc = p.weightings + static_cast<int64_t>(row) * GC::HAB(p);
      for (int t = lane; t < GC::HAB(p); t += 32) cp_async_4(sm + GC::sm_w(p) + t, wsrc + t);
    }

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
      int u0 = 0;
      for (; u0 + STEP <= cnt; u0 += STEP) {                   // full batches: no predicates
        float4 x[kFastUnroll];
        float vs[kFastUnroll];
#pragma unroll
        for (int t = 0; t < kFastUnroll; ++t) {
          const int u = u0 + t * NG + g;
          const uint32_t j = static_cast<uint32_t>(__shfl_sync(kFull, my_col, u));
          vs[t] = 0.f;
          if constexpr (MASK & P_SYM) vs[t] = __shfl_sync(kFull, my_vs, u);
          x[t] = ldg_f4_hint(src + static_cast<size_t>(j * BD), pol_keep);
        }
#pragma unroll
        for (int t = 0; t < kFastUnroll; ++t) add_edge<MASK, ARG>(acc, x[t], vs[t], e0 + u0 + t * NG + g);
      }
      if (u0 < cnt) {                                          // tail batch: loads clamped to the last nnz, adds predicated
        float4 x[kFastUnroll];
        float vs[kFastUnroll];
#pragma unroll
        for (int t = 0; t < kFastUnroll; ++t) {
          const int u = min(u0 + t * NG + g, cnt - 1);
          const uint32_t j = static_cast<uint32_t>(__shfl_sync(kFull, my_col, u));
          vs[t] = 0.f;
          if constexpr (MASK & P_SYM) vs[t] = __shfl_sync(kFull, my_vs, u);
          x[t] = ldg_f4_hint(src + static_cast<size_t>(j * BD), pol_keep);
        }
#pragma unroll
        for (int t = 0; t < kFastUnroll; ++t) {
          const int u = u0 + t * NG + g;
          if (u < cnt) add_edge<MASK, ARG>(acc, x[t], vs[t], e0 + u);
        }
      }
    }
    if constexpr (NG > 1) {
#pragma unroll
      for (int off = G; off < 32; off <<= 1) acc.merge_xor(off);
    }

    if (is_chunk) {
      // a chunk of a long row: publish the partial; the LAST chunk warp of the row to arrive merges all of them
      // in chunk order (same result whichever warp it is) and goes on to finalize the row
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
      begin = __ldg(p.rowptr + row);
      end = __ldg(p.rowptr + row + 1);
      is_chunk = false;
      if (stage_w) {
        const float* wsrc = p.weightings + static_cast<int64_t>(row) * GC::HAB(p);
        for (int t = lane; t < GC::HAB(p); t += 32) cp_async_4(sm + GC::sm_w(p) + t, wsrc + t);
      }
    }
    if (writer) {
      const bool nonempty = end > begin;
      const float cntf = static_cast<float>(max(end - begin, 1));   // mean divides by the nnz count, min 1
      const float inv = __frcp_rn(cntf);
      float mean[4] = {0.f, 0.f, 0.f, 0.f}, var[4] = {0.f, 0.f, 0.f, 0.f};
      if constexpr ((MASK & P_SUM) != 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) mean[k] = div_by(acc.sum[k], cntf, inv);
      }
      if constexpr ((MASK & P_SQ) != 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k)      // mean_sq - mean * mean, ref :242 / :271
          var[k] = __fsub_rn(div_by(acc.sq[k], cntf, inv), __fmul_rn(mean[k], mean[k]));
      }
      const size_t row_s = static_cast<size_t>(row);
#pragma unroll
      for (int a = 0; a < GC::A(p); ++a) {
        const int code = GC::aggr(p, a);
        float v[4] = {0.f, 0.f, 0.f, 0.f}, sv[4];
        int arg[4] = {-1, -1, -1, -1};
        bool gate_sign = false;
        switch (code) {
          case EGC_AGGR_SUM:
            if constexpr ((MASK & P_SUM) != 0) { for (int k = 0; k < 4; ++k) v[k] = acc.sum[k]; }
            break;
          case EGC_AGGR_MEAN:
            if constexpr ((MASK & P_SUM) != 0) { for (int k = 0; k < 4; ++k) v[k] = mean[k]; }
            break;
          case EGC_AGGR_SYMNORM:
            if constexpr ((MASK & P_SYM) != 0) { for (int k = 0; k < 4; ++k) v[k] = acc.sym[k]; }
            break;
          case EGC_AGGR_MAX:
            if constexpr ((MASK & P_MAX) != 0) {
              for (int k = 0; k < 4; ++k) { v[k] = nonempty ? acc.mx[k] : 0.f; if constexpr (ARG) arg[k] = acc.amx[k]; }
            }
            break;
          case EGC_AGGR_MIN:
            if constexpr ((MASK & P_MIN) != 0) {
              for (int k = 0; k < 4; ++k) { v[k] = nonempty ? acc.mn[k] : 0.f; if constexpr (ARG) arg[k] = acc.amn[k]; }
            }
            break;
          case EGC_AGGR_VAR:
            if constexpr ((MASK & P_SQ) != 0) { for (int k = 0; k < 4; ++k) v[k] = var[k]; }
            break;
          case EGC_AGGR_STD:
            if constexpr ((MASK & P_SQ) != 0) {       // sqrt(relu(var) + 1e-5), ref :244 / :273
              for (int k = 0; k < 4; ++k) v[k] = sqrtf(__fadd_rn(fmaxf(var[k], 0.f), kStdEps));
              gate_sign = true;
            }
            break;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) sv[k] = (gate_sign && !(var[k] > 0.f)) ? -v[k] : v[k];   // sign bit = relu gate closed
        if (p.out != nullptr) st_row<4>(sm + GC::sm_agg(p) + a * BD + foff, v);
        if (p.agg_out != nullptr) stg_f4_hint(p.agg_out + (row_s * GC::A(p) + a) * BD + foff, v, pol_stream);
        if (p.saved != nullptr) stg_f4_hint(p.saved + (row_s * GC::n_saved(p) + a) * BD + foff, sv, pol_stream);
        if constexpr (ARG) {
          const float t[4] = {__int_as_float(arg[0]), __int_as_float(arg[1]), __int_as_float(arg[2]), __int_as_float(arg[3])};
          if (p.arg_out != nullptr)
            stg_f4_hint(reinterpret_cast<float*>(p.arg_out) + (row_s * GC::A(p) + a) * BD + foff, t, pol_stream);
          if (p.saved_arg != nullptr && GC::arg_slot(p, a) >= 0)
            stg_f4_hint(reinterpret_cast<float*>(p.saved_arg) + (row_s * GC::n_arg(p) + GC::arg_slot(p, a)) * BD + foff, t, pol_stream);
        }
      }
      if constexpr ((MASK & P_SQ) != 0) {
        if (p.saved != nullptr && GC::n_saved(p) > GC::A(p)) stg_f4_hint(p.saved + (row_s * GC::n_saved(p) + GC::A(p)) * BD + foff, mean, pol_stream);
      }
    }
    if (p.out == nullptr) continue;

    // ---- per-head combination from this warp's shared memory (ref :195-208)
    cp_async_wait_all();
    __syncwarp();
    {
      const float* agg = sm + GC::sm_agg(p);
      const float* w = sm + GC::sm_w(p);
      float* out = p.out + static_cast<int64_t>(row) * GC::HD(p);
      const int D = GC::D(p), AB = GC::AB(p);
#pragma unroll
      for (int it = 0; it < kFastMaxIter; ++it) {
        const int o = lane * EV + 32 * EV * it;
        if (o < GC::HD(p)) {
          const float* wh = w + epi_w[it];
          const float* ad = agg + epi_d[it];
          if (EV == 4) {
            float r[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 12
            for (int ab = 0; ab < AB; ++ab) {
              const float wv = wh[ab];
              const float4 a = *reinterpret_cast<const float4*>(ad + ab * D);
              r[0] = fmaf(wv, a.x, r[0]); r[1] = fmaf(wv, a.y, r[1]); r[2] = fmaf(wv, a.z, r[2]); r[3] = fmaf(wv, a.w, r[3]);
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
    }
    __syncwarp();                                              // the next task overwrites this warp's staging area
  }
}

// ---------------------------------------------------------------------------------------------
// dispatch
// ---------------------------------------------------------------------------------------------
template <class Cfg, bool ARG, bool DROP = false>
int launch_fast_one(const AggParams& p, int smem_bytes, cudaStream_t st) {
  auto kern = k_aggregate_fast<Cfg, ARG, DROP>;
  if (smem_bytes > 48 * 1024) {
    EGC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  }
  const int64_t tasks = static_cast<int64_t>(p.n_chunks) + p.n_row_tasks;
  if (tasks <= 0) return EGC_OK;
  const int grid = static_cast<int>(std::min<int64_t>(ceil_div(tasks, kAggWarps), static_cast<int64_t>(sm_count()) * 4));
  {
    LaunchScope egc_ls_("k_aggregate_fwd", st);
    kern<<<grid, kAggThreads, smem_bytes, st>>>(p);
  }
  EGC_LAUNCH_CHECK("k_aggregate_fast");
  return EGC_OK;
}

template <class Cfg, bool DROP = false>
int launch_fast_arg(const AggParams& p, bool arg, int smem_bytes, cudaStream_t st) {
  if constexpr ((Cfg::MASK & (P_MAX | P_MIN)) != 0) {
    if (arg) return launch_fast_one<Cfg, true, DROP>(p, smem_bytes, st);
  }
  return launch_fast_one<Cfg, false, DROP>(p, smem_bytes, st);
}

#define EGC_FAST_MASK_CASES(X) \
  X(1) X(2) X(3) X(5) X(7) X(8) X(9) X(10) X(11) X(13) X(15) X(16) X(17) X(18) X(19) X(21) X(23) \
  X(24) X(25) X(26) X(27) X(29) X(31)

template <int G, bool DROP = false>
int launch_fast_family(const AggParams& p, int mask, bool arg, int smem_bytes, cudaStream_t st) {
  switch (mask) {
#define X(M) case M: return launch_fast_arg<DynCfg<M, G>, DROP>(p, arg, smem_bytes, st);
    EGC_FAST_MASK_CASES(X)
#undef X
  }
  set_error("aggregate: unsupported primitive mask %d", mask);
  return EGC_ERR_UNSUPPORTED;
}

}  // namespace egc
