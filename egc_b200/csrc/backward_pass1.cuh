// Backward pass 1 of the fused aggregation (per target node, streaming) and the min/max gradient routing kernel.
// Included by aggregate_api.cu only (one translation unit).
#pragma once

#include "aggregate_fast.cuh"
#include "bf16.cuh"
#include "colsum.cuh"

namespace egc {

// =============================================================================================
// backward pass 1: per target node, streaming (no graph traversal)
//   d_w[h,ab]   = sum_d g[h*D+d] * agg[ab*D+d]                       (x sigmoid' when requested)
//   d_agg[a][p] = sum_h w[h*AB + a*B + b(p)] * g[h*D + d(p)]
//   -> target-side streams t_sym / t_lin / t_sq (read by pass 2) + single-winner routing of min/max
// `saved` comes from the forward: per aggregator slot its value (std slots carry the closed relu gate
// in the sign bit), plus one extra slot with the mean when var/std is present; `saved_arg` holds the
// winning nnz position of every min/max slot.
// =============================================================================================
struct CombineBwdParams {
  const int32_t* rowptr;
  const int32_t* col;
  const float* val_lin;
  int n_rows;
  const float* weightings;
  const float* grad_out;
  const float* out_act;       // the forward's out when the layer carries the fused ReLU (grad_out is masked with out > 0), else null
  const float* epi_scale;     // [HD] scale of the forward's fused affine epilogue (the masked gradient is multiplied by it), or null
  const float* saved;
  const int32_t* saved_arg;
  float* d_weightings;
  float* tstreams;
  float* d_bases;
  int n_saved, n_arg, n_ts, ts_sym, ts_lin, ts_sq;
  int H, B, D, A, BD, HD, AB, HAB;
  int aggr[EGC_MAX_AGGR];
  int arg_slot[EGC_MAX_AGGR];
  int sigmoid;
  int sm_w, sm_g, sm_saved, sm_arg, sm_per_warp;
  int vec16;
  int64_t ts_row_stride, ts_stream_stride;   // floats between the streams of consecutive rows / between streams of a row
  float* colsum_part;                        // [grid][HD + HAB] or null
  int skip_route;                            // diagnostics: drop the min/max routing
  float* t_route;                            // [n_rows][n_arg][BD] gradients of the min/max slots, routed by k_route_minmax
};

__device__ __forceinline__ void stage_row(float* dst, const float* src, int n, int lane, bool vec16) {
  if (vec16) {
    for (int t = lane * 4; t < n; t += 128) cp_async_16(dst + t, src + t);
  } else {
    for (int t = lane; t < n; t += 32) cp_async_4(dst + t, src + t);
  }
}

constexpr int kCbColIt = 4;     // per-lane column-sum accumulators: HD <= 32 * EV * kCbColIt, HAB <= 32 * kCbColIt

__device__ __forceinline__ void stg_stream_f4(float* p, const float (&v)[4]) {
  __stcs(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
}

// Persistent warps (one target row per task).  Everything that does not depend on the row - the (head, slot)
// decomposition of a weight index, the (basis, offset) of a feature, the aggregator of a slot - is computed
// once per CTA into shared-memory tables.  The column sums of grad_out (d_bias) and of d_weightings (the
// gradient of the comb-weight bias) ride along in registers and leave as one partial row per CTA
// (deterministic: reduced in CTA order by k_colsum_partials).
// TS = storage type of the target-side streams (p.tstreams then points at bf16 rows, rounded to nearest even).
template <class Cfg, int EV, bool LINW, class TS = float>
__global__ void __launch_bounds__(kAggThreads, 4) k_combine_bwd(const __grid_constant__ CombineBwdParams p) {
  using GB = GetB<Cfg, CombineBwdParams>;
  extern __shared__ __align__(16) float smem_all[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int D = GB::D(p), BD = GB::BD(p), HD = GB::HD(p), AB = GB::AB(p), HAB = GB::HAB(p);
  // CTA-wide tables (ints) live behind the per-warp staging areas
  int* tab_goff = reinterpret_cast<int*>(smem_all + kAggWarps * GB::sm_per_warp(p));   // [HAB] h * D
  int* tab_aoff = tab_goff + HAB;                                                  // [HAB] ab * D
  int* tab_std = tab_aoff + HAB;                                                   // [HAB] slot belongs to a std aggregator
  if constexpr (!Cfg::kStatic) {
    for (int t = threadIdx.x; t < HAB; t += kAggThreads) {
      const int h = t / AB, ab = t - h * AB;
      tab_goff[t] = h * D;
      tab_aoff[t] = ab * D;
      tab_std[t] = p.aggr[ab / GB::B(p)] == EGC_AGGR_STD ? 1 : 0;
    }
    __syncthreads();
  }

  float* sm = smem_all + warp * GB::sm_per_warp(p);
  const bool v16 = p.vec16 != 0;
  const float* w = sm + GB::sm_w(p);
  const float* g = sm + GB::sm_g(p);
  const float* sv = sm + GB::sm_saved(p);
  const int nq = D >> 2;
  const int q0 = nq > 0 ? lane % nq : 0, dd0 = lane % D;
  const int warps_total = gridDim.x * kAggWarps;

  float gsum[kCbColIt][EV], wsum[kCbColIt];
#pragma unroll
  for (int it = 0; it < kCbColIt; ++it) {
    wsum[it] = 0.f;
#pragma unroll
    for (int k = 0; k < EV; ++k) gsum[it][k] = 0.f;
  }

  for (int row = blockIdx.x * kAggWarps + warp; row < p.n_rows; row += warps_total) {
    stage_row(sm + GB::sm_w(p), p.weightings + static_cast<int64_t>(row) * HAB, HAB, lane, v16);
    stage_row(sm + GB::sm_g(p), p.grad_out + static_cast<int64_t>(row) * HD, HD, lane, v16);
    stage_row(sm + GB::sm_saved(p), p.saved + static_cast<int64_t>(row) * GB::n_saved(p) * BD, GB::n_saved(p) * BD, lane, v16);
    const float cntf = static_cast<float>(max(__ldg(p.rowptr + row + 1) - __ldg(p.rowptr + row), 1));
    const float inv_cnt = __frcp_rn(cntf);
    cp_async_wait_all();
    __syncwarp();
    if (p.out_act != nullptr || p.epi_scale != nullptr) {    // fused epilogue: g <- g * (out > 0) * scale, in the staged row
      float* gs = sm + GB::sm_g(p);
      const float* oa = p.out_act != nullptr ? p.out_act + static_cast<int64_t>(row) * HD : nullptr;
      if (v16) {
        for (int t = lane * 4; t < HD; t += 128) {
          float4 gv = *reinterpret_cast<float4*>(gs + t);
          if (oa != nullptr) {
            const float4 o = __ldcs(reinterpret_cast<const float4*>(oa + t));
            gv.x = o.x > 0.f ? gv.x : 0.f; gv.y = o.y > 0.f ? gv.y : 0.f; gv.z = o.z > 0.f ? gv.z : 0.f; gv.w = o.w > 0.f ? gv.w : 0.f;
          }
          if (p.epi_scale != nullptr) {
            const float4 sc = __ldg(reinterpret_cast<const float4*>(p.epi_scale + t));
            gv.x *= sc.x; gv.y *= sc.y; gv.z *= sc.z; gv.w *= sc.w;
          }
          *reinterpret_cast<float4*>(gs + t) = gv;
        }
      } else {
        for (int t = lane; t < HD; t += 32) {
          float gv = gs[t];
          if (oa != nullptr) gv = __ldcs(oa + t) > 0.f ? gv : 0.f;
          if (p.epi_scale != nullptr) gv *= __ldg(p.epi_scale + t);
          gs[t] = gv;
        }
      }
      __syncwarp();
    }

    // (0) column sums of grad_out
    if (p.colsum_part != nullptr) {
#pragma unroll
      for (int it = 0; it < kCbColIt; ++it) {
        const int c = lane * EV + 32 * EV * it;
        if (c < HD) {
          float t[EV];
          ld_plain<EV>(t, g + c);
#pragma unroll
          for (int k = 0; k < EV; ++k) gsum[it][k] += t[k];
        }
      }
    }

    // (1) gradient of the combination weights: HAB dot products of length D, skewed start per lane
#pragma unroll
    for (int it = 0; it < kCbColIt; ++it) {
      for (int t = lane + 32 * it; t < HAB; t += 32 * kCbColIt) {
        bool is_std;
        const float* gh;
        const float* aa;
        if constexpr (Cfg::kStatic) {
          const int h = t / AB, ab = t - h * AB;
          is_std = GB::aggr(p, ab / GB::B(p)) == EGC_AGGR_STD;
          gh = g + h * D;
          aa = sv + ab * D;
        } else {
          is_std = tab_std[t] != 0;
          gh = g + tab_goff[t];
          aa = sv + tab_aoff[t];
        }
        float dot = 0.f;
        if constexpr (EV == 4) {
          int q = q0;
          for (int i = 0; i < nq; ++i) {
            const float4 gv = *reinterpret_cast<const float4*>(gh + 4 * q);
            float4 av = *reinterpret_cast<const float4*>(aa + 4 * q);
            if (is_std) { av.x = fabsf(av.x); av.y = fabsf(av.y); av.z = fabsf(av.z); av.w = fabsf(av.w); }
            dot = fmaf(gv.x, av.x, dot); dot = fmaf(gv.y, av.y, dot); dot = fmaf(gv.z, av.z, dot); dot = fmaf(gv.w, av.w, dot);
            q = (q + 1 == nq) ? 0 : q + 1;
          }
        } else {
          int dd = dd0;
          for (int i = 0; i < D; ++i) {
            const float av = is_std ? fabsf(aa[dd]) : aa[dd];
            dot = fmaf(gh[dd], av, dot);
            dd = (dd + 1 == D) ? 0 : dd + 1;
          }
        }
        if (p.sigmoid) { const float s = w[t]; dot *= s * (1.f - s); }
        __stcs(p.d_weightings + static_cast<int64_t>(row) * HAB + t, dot);
        if (t < 32 * kCbColIt) wsum[it] += dot;
      }
    }

    // (2) gradient w.r.t. the aggregates -> target-side streams and min/max routing
    TS* ts = reinterpret_cast<TS*>(p.tstreams) + static_cast<int64_t>(row) * p.ts_row_stride;
    for (int p0 = lane * EV; p0 < BD; p0 += 32 * EV) {
      const int b = p0 / D, d = p0 - b * D;
      float t_sym[EV], t_lin[EV], t_sq[EV];
#pragma unroll
      for (int k = 0; k < EV; ++k) { t_sym[k] = 0.f; t_lin[k] = 0.f; t_sq[k] = 0.f; }
#pragma unroll
      for (int a = 0; a < GB::A(p); ++a) {
        float da[EV];
#pragma unroll
        for (int k = 0; k < EV; ++k) da[k] = 0.f;
        const float* wa = w + a * GB::B(p) + b;
#pragma unroll
        for (int h = 0; h < GB::H(p); ++h) {
          const float wv = wa[h * AB];
          float gv[EV];
          ld_plain<EV>(gv, g + h * D + d);
#pragma unroll
          for (int k = 0; k < EV; ++k) da[k] = fmaf(wv, gv[k], da[k]);
        }
        const int code = GB::aggr(p, a);
        if (code == EGC_AGGR_SUM) {
#pragma unroll
          for (int k = 0; k < EV; ++k) t_lin[k] += da[k];
        } else if (code == EGC_AGGR_MEAN) {
#pragma unroll
          for (int k = 0; k < EV; ++k) t_lin[k] = fmaf(da[k], inv_cnt, t_lin[k]);
        } else if (code == EGC_AGGR_SYMNORM) {
#pragma unroll
          for (int k = 0; k < EV; ++k) t_sym[k] += da[k];
        } else if (code == EGC_AGGR_MAX || code == EGC_AGGR_MIN) {
          // routed to the single winning source by k_route_minmax (feature-slab order keeps its atomics in the L2)
          float* tr = p.t_route + (static_cast<int64_t>(row) * GB::n_arg(p) + GB::arg_slot(p, a)) * BD + p0;
          if constexpr (EV == 4) stg_stream_f4(tr, da); else st_row<EV>(tr, da);
        } else {   // VAR / STD
          float sa[EV], mean[EV];
          ld_plain<EV>(sa, sv + a * BD + p0);
          ld_plain<EV>(mean, sv + GB::A(p) * BD + p0);
#pragma unroll
          for (int k = 0; k < EV; ++k) {
            float dv = da[k];
            if (code == EGC_AGGR_STD) dv = sa[k] > 0.f ? __fdividef(dv, 2.f * sa[k]) : 0.f;    // relu gate (sign bit), d sqrt
            const float q = dv * inv_cnt;
            t_sq[k] += q;
            t_lin[k] = fmaf(-2.f * mean[k], q, t_lin[k]);
          }
        }
      }
      // plain (L2 write-back) stores: pass 2 gathers these rows next, whatever part of them survives in the L2 is a hit
      TS* tsp = ts + p0;
      if constexpr (kBf16<TS>) {
        auto st_ts = [&](TS* q, const float (&v)[EV]) {
          if constexpr (EV == 4) st4<TS>(q, v); else st1<TS>(q, v[0]);
        };
        if (GB::ts_sym(p) >= 0) st_ts(tsp + static_cast<int64_t>(GB::ts_sym(p)) * p.ts_stream_stride, t_sym);
        if (GB::ts_lin(p) >= 0) st_ts(tsp + static_cast<int64_t>(GB::ts_lin(p)) * p.ts_stream_stride, t_lin);
        if (GB::ts_sq(p) >= 0) st_ts(tsp + static_cast<int64_t>(GB::ts_sq(p)) * p.ts_stream_stride, t_sq);
      } else {
        if (GB::ts_sym(p) >= 0) st_row<EV>(tsp + static_cast<int64_t>(GB::ts_sym(p)) * p.ts_stream_stride, t_sym);
        if (GB::ts_lin(p) >= 0) st_row<EV>(tsp + static_cast<int64_t>(GB::ts_lin(p)) * p.ts_stream_stride, t_lin);
        if (GB::ts_sq(p) >= 0) st_row<EV>(tsp + static_cast<int64_t>(GB::ts_sq(p)) * p.ts_stream_stride, t_sq);
      }
    }
    __syncwarp();     // the next row overwrites this warp's staging area
  }

  // ---- column-sum partials of this CTA: [HD] grad_out sums | [HAB] d_weightings sums
  if (p.colsum_part != nullptr) {
    __syncthreads();
    float* red = smem_all;                                   // reuse the staging areas: [kAggWarps][HD + HAB]
    const int width = HD + HAB;
#pragma unroll
    for (int it = 0; it < kCbColIt; ++it) {
      const int c = lane * EV + 32 * EV * it;
      if (c < HD) {
#pragma unroll
        for (int k = 0; k < EV; ++k) red[warp * width + c + k] = gsum[it][k];
      }
      const int t = lane + 32 * it;
      if (t < HAB) red[warp * width + HD + t] = wsum[it];
    }
    __syncthreads();
    for (int c = threadIdx.x; c < width; c += kAggThreads) {
      float t = 0.f;
#pragma unroll
      for (int wv = 0; wv < kAggWarps; ++wv) t += red[wv * width + c];
      p.colsum_part[static_cast<int64_t>(blockIdx.x) * width + c] = t;
    }
  }
}

// out[c] = sum over CTAs of part[cta][c] in CTA order; columns [0, n1) -> out1, [n1, n1 + n2) -> out2
__global__ void k_colsum_partials(const float* __restrict__ part, int n_cta, int n1, int n2, float* __restrict__ out1,
                                  float* __restrict__ out2) {
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int width = n1 + n2;
  if (c >= width) return;
  float t = 0.f;
  for (int s = lane; s < n_cta; s += 32) t += part[static_cast<int64_t>(s) * width + c];
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(kFull, t, o);
  if (lane == 0) {
    if (c < n1) { if (out1 != nullptr) out1[c] = t; }
    else if (out2 != nullptr) out2[c - n1] = t;
  }
}


// =============================================================================================
// min/max gradient routing: d_bases[col[arg[i][s][p]]][p] += t_route[i][s][p]   (x val_lin[arg] when weighted)
// One warp task = 32 consecutive features of kRouteRows consecutive target rows.  The grid walks the
// (feature slab, slot) phases together, so at any moment it adds into one 32-float column slab of d_bases
// (n_src x 128 B - L2-resident) instead of missing to DRAM all over the [n_src, BD] matrix.
// Hub sources (the long columns of the CSC plan: a power-law hub sits in thousands of rows and wins a share of
// the features in each) would serialise tens of thousands of fp32 REDs on ONE 128-byte line per phase - the L2
// atomic unit retires about one lane per cycle per line - so every CTA privatises them: a shared-memory hash
// maps the hub ids to slots, their contributions go to shared-memory accumulators (ATOMS), and each CTA flushes
// one RED per (hub, feature) at the end of the phase.
// =============================================================================================
constexpr int kRouteRows = 8;
constexpr int kRouteThreads = 1024;
constexpr int kRouteMaxHubs = 1024;
constexpr int kRouteHashSize = 2 * kRouteMaxHubs;           // open addressing, load factor <= 0.5

struct RouteParams {
  const int32_t* saved_arg;    // [n_rows][n_arg][BD] winning nnz position (-1: none)
  const float* t_route;        // [n_rows][n_arg][BD]
  const int32_t* col;
  const float* val_lin;        // or null
  float* d_bases;              // [n_src][BD]
  const int32_t* hubs;         // [n_hubs] source ids privatised in shared memory (or null)
  int n_hubs;
  int n_rows, n_arg, BD, n_slabs;
};

__device__ __forceinline__ uint32_t route_hash(int j) { return (static_cast<uint32_t>(j) * 2654435761u) >> (32 - 11); }
static_assert(kRouteHashSize == 1 << 11, "route_hash yields 11 bits");

__global__ void __launch_bounds__(kRouteThreads, 1) k_route_minmax(const __grid_constant__ RouteParams p) {
  extern __shared__ __align__(16) float route_smem[];
  int* hash_key = reinterpret_cast<int*>(route_smem);                       // [kRouteHashSize] source id or -1
  int* hash_slot = hash_key + kRouteHashSize;                               // [kRouteHashSize]
  float* acc = reinterpret_cast<float*>(hash_slot + kRouteHashSize);        // [n_hubs][32]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int warps_cta = blockDim.x >> 5;
  const int warps_total = gridDim.x * warps_cta;
  const int row_groups = (p.n_rows + kRouteRows - 1) / kRouteRows;
  const int64_t row_stride = static_cast<int64_t>(p.n_arg) * p.BD;
  const bool hubs_on = p.n_hubs > 0;
  if (hubs_on) {
    for (int t = threadIdx.x; t < kRouteHashSize; t += blockDim.x) hash_key[t] = -1;
    for (int t = threadIdx.x; t < p.n_hubs * 32; t += blockDim.x) acc[t] = 0.f;
    __syncthreads();
    for (int t = threadIdx.x; t < p.n_hubs; t += blockDim.x) {
      const int j = __ldg(p.hubs + t);
      uint32_t h = route_hash(j);
      while (atomicCAS(hash_key + h, -1, j) != -1) h = (h + 1) & (kRouteHashSize - 1);   // hub ids are distinct
      hash_slot[h] = t;
    }
    __syncthreads();
  }
  for (int phase = 0; phase < p.n_slabs * p.n_arg; ++phase) {
    const int slab = phase / p.n_arg, slot = phase - slab * p.n_arg;
    const int f = slab * 32 + lane;
    const bool f_ok = f < p.BD;
    const int64_t base = static_cast<int64_t>(slot) * p.BD + f;
    for (int rg = blockIdx.x * warps_cta + warp; rg < row_groups; rg += warps_total) {
      int arg[kRouteRows];
      float v[kRouteRows];
#pragma unroll
      for (int r = 0; r < kRouteRows; ++r) {
        const int row = rg * kRouteRows + r;
        arg[r] = -1;
        v[r] = 0.f;
        if (row < p.n_rows && f_ok) {
          arg[r] = __ldcs(p.saved_arg + row * row_stride + base);
          v[r] = __ldcs(p.t_route + row * row_stride + base);
        }
      }
      int j[kRouteRows];
#pragma unroll
      for (int r = 0; r < kRouteRows; ++r) {
        j[r] = arg[r] >= 0 ? __ldg(p.col + arg[r]) : -1;
        if (p.val_lin != nullptr && arg[r] >= 0) v[r] *= __ldg(p.val_lin + arg[r]);
      }
#pragma unroll
      for (int r = 0; r < kRouteRows; ++r) {
        if (j[r] < 0) continue;
        int hub = -1;
        if (hubs_on) {
          uint32_t h = route_hash(j[r]);
          int k = hash_key[h];
          while (k != -1 && k != j[r]) { h = (h + 1) & (kRouteHashSize - 1); k = hash_key[h]; }
          if (k == j[r]) hub = hash_slot[h];
        }
        if (hub >= 0) atomicAdd(acc + hub * 32 + lane, v[r]);
        else atomicAdd(p.d_bases + static_cast<int64_t>(j[r]) * p.BD + f, v[r]);
      }
    }
    if (hubs_on) {                                           // flush this CTA's hub partials of the phase
      __syncthreads();
      for (int t = threadIdx.x; t < p.n_hubs * 32; t += blockDim.x) {
        const float a = acc[t];
        const int ff = slab * 32 + (t & 31);
        if (a != 0.f && ff < p.BD) atomicAdd(p.d_bases + static_cast<int64_t>(__ldg(p.hubs + (t >> 5))) * p.BD + ff, a);
        acc[t] = 0.f;
      }
      __syncthreads();
    }
  }
}


}  // namespace egc
