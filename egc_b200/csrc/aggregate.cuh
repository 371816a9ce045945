// Fused multi-aggregator CSR SpMM + combination: shared device machinery (sm_100a).
//
// One warp owns one task: a whole CSR row (<= EGC_CHUNK_EDGES nnz), one chunk of a long row, or the
// merge of a long row's chunk partials.  A basis row (B*D floats) is spread over the lanes of a
// "group" of G lanes in VEC-wide pieces (VEC = 4 -> 128-bit gathers); when the row is narrower than
// 32*VEC floats the warp's 32/G groups walk different neighbours in parallel and are merged with
// xor-shuffles at the end.  All requested aggregators are produced from ONE gather of each
// neighbour row: primitives sum / symnorm-sum / sum of squares / max(+arg) / min(+arg).
//
// The gather loop is branch-free: a batch of kGatherUnroll neighbours is always issued; slots past
// the end of the row re-read the row's last neighbour (harmless for max/min, which keep the first
// winner) and carry weight 0 into the sums.
#pragma once

#include <float.h>

#include "common.cuh"

namespace egc {

enum Prim : int { P_SUM = 1, P_SYM = 2, P_SQ = 4, P_MAX = 8, P_MIN = 16 };

constexpr int kAggWarps = 8;
constexpr int kAggThreads = kAggWarps * 32;
constexpr int kGatherUnroll = 8;      // independent 128-bit gathers in flight per lane
constexpr float kStdEps = 1e-5f;      // ref optimized_layers.py:244,273

struct AggParams {
  // target-major CSR
  const int32_t* rowptr;
  const int32_t* col;
  const float* val_sym;
  const float* val_lin;
  int n_rows;
  const int32_t* row_map;    // optional subset of rows handled as row tasks (null: all rows)
  int n_row_tasks;
  // long-row plan + scratch for chunk partials [n_chunks][n_slots][BD]
  int n_long, n_chunks;
  const int32_t* long_rows;
  const int32_t* long_chunk_ptr;
  const int32_t* chunk_row;
  const int32_t* chunk_begin;
  float* partials;
  int n_slots;
  int* long_counter;         // [n_long] zero on entry: chunk warps count in, the last one merges (fast kernel)
  // features
  const float* bases;        // [n_src, BD]
  const float* weightings;   // [n_rows, HAB]
  const float* bias;         // [HD] or null
  const float* epi_scale;    // fused epilogue (egc_epilogue): y = y * scale + shift, [HD] each, or null
  const float* epi_shift;
  const float* epi_add;      // [n_rows, HD] added after the activation, or null (may alias out)
  const float* agg_init;     // [n_rows, A, BD] partial aggregates of an earlier call over another entry subset (sum / symnorm
                             // only), added to this call's before saving / combining; or null (may alias agg_out / saved)
  float* out;                // [n_rows, HD] or null
  float* agg_out;            // [n_rows, A, BD] or null   (reference `aggregated`)
  int32_t* arg_out;          // [n_rows, A, BD] or null
  float* saved;              // [n_rows, S, BD] or null   (training: what the backward needs)
  int32_t* saved_arg;        // [n_rows, n_arg, BD] or null
  int n_saved, n_arg;        // S = A (+1 mean slot when var/std present); n_arg = # of min/max slots
  // shape
  int H, B, D, A, BD, HD, AB, HAB;
  int aggr[EGC_MAX_AGGR];
  int arg_slot[EGC_MAX_AGGR];   // index into saved_arg for min/max aggregators, else -1
  int sigmoid;
  int relu;      // fused output activation: out = max(out, 0)
  // lane geometry
  int nvec;      // VEC-wide pieces per basis row
  int G;         // lanes per group (power of two, <= 32)
  int n_pass;    // passes of 32 pieces when nvec > 32
  // per-warp shared memory layout (float offsets)
  int sm_agg, sm_w, sm_per_warp;
  int mode;      // 0: chunk tasks then row tasks, 1: merge tasks (one per long row)
  int rows_per_task;   // row-block kernel: consecutive rows per task (<= EGC_ROWS_PER_TASK); fewer when the launch is small
  // fused dropout after the ReLU (egc_dropout), read only by the kernels instantiated with DROP = true: keep (row, c) iff
  // Philox4x32-10 word c & 3 of counter (c >> 2, drop_row0 + row, 0, 0) under key *drop_seed is < drop_thresh; kept
  // values are scaled by drop_scale
  const uint64_t* drop_seed;   // null: no dropout
  uint32_t drop_thresh;
  float drop_scale;
  int64_t drop_row0;           // global id of local row 0
};

// ---------------------------------------------------------------------------------------------
// vector load / store of VEC consecutive floats
// ---------------------------------------------------------------------------------------------
template <int VEC>
__device__ __forceinline__ void ld_row(float (&v)[VEC], const float* __restrict__ p) {
  if constexpr (VEC == 4) {
    float4 t = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else {
#pragma unroll
    for (int k = 0; k < VEC; ++k) v[k] = __ldg(p + k);
  }
}

template <int VEC>
__device__ __forceinline__ void ld_plain(float (&v)[VEC], const float* p) {
  if constexpr (VEC == 4) {
    float4 t = *reinterpret_cast<const float4*>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else {
#pragma unroll
    for (int k = 0; k < VEC; ++k) v[k] = p[k];
  }
}

// L2-only load (data written by other SMs during this kernel)
template <int VEC>
__device__ __forceinline__ void ld_cg(float (&v)[VEC], const float* p) {
  if constexpr (VEC == 4) {
    float4 t = __ldcg(reinterpret_cast<const float4*>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else {
#pragma unroll
    for (int k = 0; k < VEC; ++k) v[k] = __ldcg(p + k);
  }
}

template <int VEC>
__device__ __forceinline__ void st_row(float* p, const float (&v)[VEC]) {
  if constexpr (VEC == 4) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
#pragma unroll
    for (int k = 0; k < VEC; ++k) p[k] = v[k];
  }
}

// streaming (evict-first) store: outputs that are not re-read by this kernel
template <int VEC>
__device__ __forceinline__ void st_stream(float* p, const float (&v)[VEC]) {
  if constexpr (VEC == 4) {
    __stcs(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
  } else {
#pragma unroll
    for (int k = 0; k < VEC; ++k) __stcs(p + k, v[k]);
  }
}

__device__ __forceinline__ void cp_async_4(void* smem_dst, const void* gmem_src) {
  unsigned d = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(d), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gmem_src) {
  unsigned d = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// fused dropout: Philox4x32-10 (Salmon et al., SC'11; the Random123 constants), one call per 4 output columns
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r > 0) { k.x += 0x9E3779B9u; k.y += 0xBB67AE85u; }
    const uint32_t lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const uint32_t lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
  }
  return c;
}

// keep bits of columns 4q .. 4q + 3 of global row `grow` (bit w = column 4q + w).  Out of line, and the key is read here
// (an L1-resident word): the forward kernels run at their register caps, and a key held from kernel start, or the
// Philox rounds inlined into the epilogue loops, made the dropout instantiations spill in their gather loops
static __device__ __noinline__ uint32_t dropout_keep4(const uint64_t* seed, uint32_t thresh, uint32_t q, uint32_t grow) {
  const uint64_t s = __ldg(reinterpret_cast<const unsigned long long*>(seed));
  const uint4 u = philox4x32_10(make_uint4(q, grow, 0u, 0u), make_uint2(static_cast<uint32_t>(s), static_cast<uint32_t>(s >> 32)));
  return (u.x < thresh ? 1u : 0u) | (u.y < thresh ? 2u : 0u) | (u.z < thresh ? 4u : 0u) | (u.w < thresh ? 8u : 0u);
}

// columns c0 .. c0 + 3 (c0 % 4 == 0) of local row `row`, after the ReLU
__device__ __forceinline__ void dropout4(const AggParams& p, float (&r)[4], int64_t row, int c0) {
  const uint32_t m = dropout_keep4(p.drop_seed, p.drop_thresh, static_cast<uint32_t>(c0) >> 2, static_cast<uint32_t>(p.drop_row0 + row));
#pragma unroll
  for (int w = 0; w < 4; ++w) r[w] = (m >> w) & 1u ? __fmul_rn(r[w], p.drop_scale) : 0.f;
}
// one column (the scalar tails, D % 4 != 0): the same word of the same draw
__device__ __forceinline__ float dropout1(const AggParams& p, float r, int64_t row, int c) {
  const uint32_t m = dropout_keep4(p.drop_seed, p.drop_thresh, static_cast<uint32_t>(c) >> 2, static_cast<uint32_t>(p.drop_row0 + row));
  return (m >> (c & 3)) & 1u ? __fmul_rn(r, p.drop_scale) : 0.f;
}

// ---------------------------------------------------------------------------------------------
// accumulator of the aggregation primitives for VEC features
// ---------------------------------------------------------------------------------------------
template <int MASK, int VEC, bool LINW, bool ARG>
struct Acc {
  float sum[VEC], sym[VEC], sq[VEC], mx[VEC], mn[VEC];
  int amx[VEC], amn[VEC];

  __device__ __forceinline__ void init() {
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      sum[k] = 0.f; sym[k] = 0.f; sq[k] = 0.f;
      mx[k] = -INFINITY; mn[k] = INFINITY;
      amx[k] = -1; amn[k] = -1;
    }
  }

  // One neighbour.  m = 1 for a real neighbour, 0 for a padding slot (which re-reads the last real one);
  // vs = its symnorm weight (0 for padding); vl = its linear weight (LINW only); e = nnz position.
  // Products and sums are rounded separately (no FMA contraction of x*w + s), so a sequential walk
  // reproduces the reference's fp32 results bit for bit.
  __device__ __forceinline__ void add(const float (&x)[VEC], float m, float vs, float vl, int e) {
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      const float msg = LINW ? __fmul_rn(x[k], vl) : x[k];          // message seen by sum/mean/min/max/var
      if constexpr (MASK & P_SUM) sum[k] = fmaf(msg, m, sum[k]);     // exact: m is 0 or 1
      if constexpr (MASK & P_SQ) {
        float s = __fmul_rn(x[k], x[k]);
        if (LINW) s = __fmul_rn(s, vl);
        sq[k] = fmaf(s, m, sq[k]);
      }
      if constexpr (MASK & P_SYM) sym[k] = __fadd_rn(sym[k], __fmul_rn(x[k], vs));
      if constexpr (MASK & P_MAX) {
        if constexpr (ARG) { if (msg > mx[k]) { mx[k] = msg; amx[k] = e; } }
        else mx[k] = fmaxf(mx[k], msg);
      }
      if constexpr (MASK & P_MIN) {
        if constexpr (ARG) { if (msg < mn[k]) { mn[k] = msg; amn[k] = e; } }
        else mn[k] = fminf(mn[k], msg);
      }
    }
  }

  // ties between partial results: the smaller nnz position wins (-1 = empty compares as +inf)
  __device__ __forceinline__ void merge_max(int k, float o, int oa) {
    if constexpr (ARG) {
      if (o > mx[k] || (o == mx[k] && static_cast<unsigned>(oa) < static_cast<unsigned>(amx[k]))) { mx[k] = o; amx[k] = oa; }
    } else {
      mx[k] = fmaxf(mx[k], o);
    }
  }
  __device__ __forceinline__ void merge_min(int k, float o, int oa) {
    if constexpr (ARG) {
      if (o < mn[k] || (o == mn[k] && static_cast<unsigned>(oa) < static_cast<unsigned>(amn[k]))) { mn[k] = o; amn[k] = oa; }
    } else {
      mn[k] = fminf(mn[k], o);
    }
  }

  __device__ __forceinline__ void merge_xor(int off) {
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      if constexpr (MASK & P_SUM) sum[k] = __fadd_rn(sum[k], __shfl_xor_sync(kFull, sum[k], off));
      if constexpr (MASK & P_SYM) sym[k] = __fadd_rn(sym[k], __shfl_xor_sync(kFull, sym[k], off));
      if constexpr (MASK & P_SQ) sq[k] = __fadd_rn(sq[k], __shfl_xor_sync(kFull, sq[k], off));
      if constexpr (MASK & P_MAX) {
        float o = __shfl_xor_sync(kFull, mx[k], off);
        int oa = ARG ? __shfl_xor_sync(kFull, amx[k], off) : 0;
        merge_max(k, o, oa);
      }
      if constexpr (MASK & P_MIN) {
        float o = __shfl_xor_sync(kFull, mn[k], off);
        int oa = ARG ? __shfl_xor_sync(kFull, amn[k], off) : 0;
        merge_min(k, o, oa);
      }
    }
  }

  // partial <-> scratch; `p` points at slot 0 of this lane's features, slots are BD floats apart.
  // Slot order: SUM, SYM, SQ, MAX, AMAX, MIN, AMIN (arg slots always reserved, see n_slots_of_mask).
  __device__ __forceinline__ void store(float* p, int BD) const {
    int s = 0;
    if constexpr (MASK & P_SUM) { st_row<VEC>(p + s * BD, sum); ++s; }
    if constexpr (MASK & P_SYM) { st_row<VEC>(p + s * BD, sym); ++s; }
    if constexpr (MASK & P_SQ) { st_row<VEC>(p + s * BD, sq); ++s; }
    if constexpr (MASK & P_MAX) {
      st_row<VEC>(p + s * BD, mx); ++s;
      if constexpr (ARG) {
        float t[VEC];
#pragma unroll
        for (int k = 0; k < VEC; ++k) t[k] = __int_as_float(amx[k]);
        st_row<VEC>(p + s * BD, t);
      }
      ++s;
    }
    if constexpr (MASK & P_MIN) {
      st_row<VEC>(p + s * BD, mn); ++s;
      if constexpr (ARG) {
        float t[VEC];
#pragma unroll
        for (int k = 0; k < VEC; ++k) t[k] = __int_as_float(amn[k]);
        st_row<VEC>(p + s * BD, t);
      }
      ++s;
    }
  }

  __device__ __forceinline__ void merge_from(const float* p, int BD) {
    int s = 0;
    float t[VEC], u[VEC];
    if constexpr (MASK & P_SUM) {
      ld_cg<VEC>(t, p + s * BD); ++s;
#pragma unroll
      for (int k = 0; k < VEC; ++k) sum[k] = __fadd_rn(sum[k], t[k]);
    }
    if constexpr (MASK & P_SYM) {
      ld_cg<VEC>(t, p + s * BD); ++s;
#pragma unroll
      for (int k = 0; k < VEC; ++k) sym[k] = __fadd_rn(sym[k], t[k]);
    }
    if constexpr (MASK & P_SQ) {
      ld_cg<VEC>(t, p + s * BD); ++s;
#pragma unroll
      for (int k = 0; k < VEC; ++k) sq[k] = __fadd_rn(sq[k], t[k]);
    }
    if constexpr (MASK & P_MAX) {
      ld_cg<VEC>(t, p + s * BD); ++s;
#pragma unroll
      for (int k = 0; k < VEC; ++k) u[k] = 0.f;
      if constexpr (ARG) ld_cg<VEC>(u, p + s * BD);
      ++s;
#pragma unroll
      for (int k = 0; k < VEC; ++k) merge_max(k, t[k], __float_as_int(u[k]));
    }
    if constexpr (MASK & P_MIN) {
      ld_cg<VEC>(t, p + s * BD); ++s;
#pragma unroll
      for (int k = 0; k < VEC; ++k) u[k] = 0.f;
      if constexpr (ARG) ld_cg<VEC>(u, p + s * BD);
      ++s;
#pragma unroll
      for (int k = 0; k < VEC; ++k) merge_min(k, t[k], __float_as_int(u[k]));
    }
  }
};

// ---------------------------------------------------------------------------------------------
// walk nnz [begin, end) of one row; lanes of group g = lane / G take neighbours g, g + NG, ...
// `foff` must be a valid feature offset for every lane (inactive lanes are clamped by the caller).
// ---------------------------------------------------------------------------------------------
template <int MASK, int VEC, bool LINW, bool ARG>
__device__ __forceinline__ void accumulate_range(Acc<MASK, VEC, LINW, ARG>& acc, const AggParams& p, int begin,
                                                 int end, int lane, int foff) {
  const int G = p.G, NG = 32 / G, g = lane / G;
  const float* __restrict__ src = p.bases + foff;
  const int64_t stride = p.BD;
  const int last = end - 1;
  for (int e0 = begin + g; e0 < end + g; e0 += kGatherUnroll * NG) {   // e0 - g is warp-uniform
    int ec[kGatherUnroll], j[kGatherUnroll];
    float m[kGatherUnroll], vs[kGatherUnroll], vl[kGatherUnroll];
#pragma unroll
    for (int u = 0; u < kGatherUnroll; ++u) {
      const int e = e0 + u * NG;
      ec[u] = min(e, last);
      m[u] = e <= last ? 1.f : 0.f;
      j[u] = __ldg(p.col + ec[u]);
      vs[u] = 0.f; vl[u] = 1.f;
      if constexpr (MASK & P_SYM) vs[u] = e <= last ? __ldg(p.val_sym + ec[u]) : 0.f;
      if constexpr (LINW) vl[u] = __ldg(p.val_lin + ec[u]);
    }
    float x[kGatherUnroll][VEC];
#pragma unroll
    for (int u = 0; u < kGatherUnroll; ++u) ld_row<VEC>(x[u], src + j[u] * stride);
#pragma unroll
    for (int u = 0; u < kGatherUnroll; ++u) acc.add(x[u], m[u], vs[u], vl[u], ec[u]);
  }
  for (int off = G; off < 32; off <<= 1) acc.merge_xor(off);
}

// value of aggregator `code` for feature k of this lane, from the primitives
template <int MASK, int VEC, bool LINW, bool ARG>
__device__ __forceinline__ float finalize_one(const Acc<MASK, VEC, LINW, ARG>& acc, int code, int k, float cntf,
                                              bool nonempty, float& mean_out, float& var_out) {
  switch (code) {
    case EGC_AGGR_SUM:
      if constexpr (MASK & P_SUM) return acc.sum[k];
      break;
    case EGC_AGGR_MEAN:
      if constexpr (MASK & P_SUM) return __fdiv_rn(acc.sum[k], cntf);
      break;
    case EGC_AGGR_SYMNORM:
      if constexpr (MASK & P_SYM) return acc.sym[k];
      break;
    case EGC_AGGR_MAX:
      if constexpr (MASK & P_MAX) return nonempty ? acc.mx[k] : 0.f;     // empty row -> 0
      break;
    case EGC_AGGR_MIN:
      if constexpr (MASK & P_MIN) return nonempty ? acc.mn[k] : 0.f;
      break;
    case EGC_AGGR_VAR:
    case EGC_AGGR_STD:
      if constexpr ((MASK & P_SQ) && (MASK & P_SUM)) {
        const float mean = __fdiv_rn(acc.sum[k], cntf);
        const float msq = __fdiv_rn(acc.sq[k], cntf);
        const float var = __fsub_rn(msq, __fmul_rn(mean, mean));   // mean_sq - mean*mean, ref :242 / :271
        mean_out = mean;
        var_out = var;
        if (code == EGC_AGGR_VAR) return var;
        return sqrtf(__fadd_rn(fmaxf(var, 0.f), kStdEps));          // sqrt(relu(var) + 1e-5), ref :244 / :273
      }
      break;
  }
  return 0.f;
}

inline int prim_mask_of(const egc_layer_desc& d) {
  int m = 0;
  for (int a = 0; a < d.n_aggr; ++a) {
    switch (d.aggr[a]) {
      case EGC_AGGR_SUM: case EGC_AGGR_MEAN: m |= P_SUM; break;
      case EGC_AGGR_SYMNORM: m |= P_SYM; break;
      case EGC_AGGR_MAX: m |= P_MAX; break;
      case EGC_AGGR_MIN: m |= P_MIN; break;
      case EGC_AGGR_VAR: case EGC_AGGR_STD: m |= P_SUM | P_SQ; break;
      default: return -1;
    }
  }
  return m;
}

inline int n_slots_of_mask(int m) {
  return ((m & P_SUM) ? 1 : 0) + ((m & P_SYM) ? 1 : 0) + ((m & P_SQ) ? 1 : 0) + ((m & P_MAX) ? 2 : 0) +
         ((m & P_MIN) ? 2 : 0);
}

inline bool has_var_like(const egc_layer_desc& d) {
  for (int a = 0; a < d.n_aggr; ++a)
    if (d.aggr[a] == EGC_AGGR_VAR || d.aggr[a] == EGC_AGGR_STD) return true;
  return false;
}
inline int n_arg_slots(const egc_layer_desc& d) {
  int n = 0;
  for (int a = 0; a < d.n_aggr; ++a) n += (d.aggr[a] == EGC_AGGR_MAX || d.aggr[a] == EGC_AGGR_MIN) ? 1 : 0;
  return n;
}
inline int n_saved_slots(const egc_layer_desc& d) { return d.n_aggr + (has_var_like(d) ? 1 : 0); }

// host: fill shape / geometry / smem layout fields; returns dynamic smem bytes per CTA
int fill_agg_params(AggParams& p, const egc_layer_desc& d, bool vec4);

// launchers (one translation unit per VEC/ARG combination to keep compile times parallel).  The *_dropout launchers run the
// same kernels instantiated with DROP = true (fused dropout after the ReLU, p.drop_seed != null; *_dropout.cu); every
// other launch runs kernels without a line of dropout code
int launch_aggregate_v4(const AggParams& p, int mask, bool linw, bool arg, int smem_bytes, cudaStream_t st);
int launch_aggregate_v1(const AggParams& p, int mask, bool linw, bool arg, int smem_bytes, cudaStream_t st);
// fast path (aggregate_fast.cuh): vec4 rows of <= 128 floats, no per-nnz linear weights, mode 0 only
int launch_aggregate_fast_g32(const AggParams& p, int mask, bool arg, int smem_bytes, cudaStream_t st);
int launch_aggregate_fast_g16(const AggParams& p, int mask, bool arg, int smem_bytes, cudaStream_t st);
// fast path with heads / bases / head dim / aggregator list baked in (aggregate_fast_static.cu); cfg_index from static_cfg_index()
int launch_aggregate_fast_static(int cfg_index, const AggParams& p, bool arg, int smem_bytes, cudaStream_t st);
// row-block kernel (aggregate_rows.cuh): whole-graph calls of the specialised layer shapes; *task_counter must be 0
int launch_aggregate_rows_static(int cfg_index, const AggParams& p, bool arg, int* task_counter, cudaStream_t st);
int launch_aggregate_rows_g32(const AggParams& p, int mask, bool arg, int* task_counter, cudaStream_t st);
int launch_aggregate_rows_g16(const AggParams& p, int mask, bool arg, int* task_counter, cudaStream_t st);
int rows_kernel_smem_bytes(const AggParams& p);
// the same kernel over bf16 basis rows (p.bases -> bf16, p.nvec = B*D / 8; aggregate_rows_bf16_*.cu)
int launch_aggregate_rows_bf16_static(int cfg_index, const AggParams& p, bool arg, int* task_counter, cudaStream_t st);
int launch_aggregate_rows_bf16_g8(const AggParams& p, int mask, bool arg, int* task_counter, cudaStream_t st);
int launch_aggregate_rows_bf16_g16(const AggParams& p, int mask, bool arg, int* task_counter, cudaStream_t st);
int launch_aggregate_v4_dropout(const AggParams& p, int mask, bool linw, bool arg, int smem_bytes, cudaStream_t st);
int launch_aggregate_v1_dropout(const AggParams& p, int mask, bool linw, bool arg, int smem_bytes, cudaStream_t st);
int launch_aggregate_fast_g32_dropout(const AggParams& p, int mask, bool arg, int smem_bytes, cudaStream_t st);
int launch_aggregate_fast_g16_dropout(const AggParams& p, int mask, bool arg, int smem_bytes, cudaStream_t st);
int launch_aggregate_fast_static_dropout(int cfg_index, const AggParams& p, bool arg, int smem_bytes, cudaStream_t st);
int launch_aggregate_rows_static_dropout(int cfg_index, const AggParams& p, bool arg, int* task_counter, cudaStream_t st);
int launch_aggregate_rows_g32_dropout(const AggParams& p, int mask, bool arg, int* task_counter, cudaStream_t st);
int launch_aggregate_rows_g16_dropout(const AggParams& p, int mask, bool arg, int* task_counter, cudaStream_t st);
int launch_aggregate_rows_bf16_static_dropout(int cfg_index, const AggParams& p, bool arg, int* task_counter, cudaStream_t st);
int launch_aggregate_rows_bf16_g8_dropout(const AggParams& p, int mask, bool arg, int* task_counter, cudaStream_t st);
int launch_aggregate_rows_bf16_g16_dropout(const AggParams& p, int mask, bool arg, int* task_counter, cudaStream_t st);

}  // namespace egc
