// extern "C" entry points of the fused aggregation forward / backward: argument validation, workspace layout, kernel
// selection.  The backward kernels live in backward_pass1.cuh (per-target streaming pass, min/max routing) and
// backward_pass2.cuh (per-source CSC gather pass); the forward kernels in aggregate_rows.cuh / aggregate_fast.cuh /
// aggregate_impl.cuh.
#include <stdlib.h>

#include <algorithm>
#include <cmath>

#include "aggregate_fast.cuh"
#include "colsum.cuh"

namespace egc {

int fill_agg_params(AggParams& p, const egc_layer_desc& d, bool vec4) {
  p.H = d.heads; p.B = d.bases; p.D = d.dim; p.A = d.n_aggr;
  p.BD = d.bases * d.dim; p.HD = d.heads * d.dim; p.AB = d.n_aggr * d.bases; p.HAB = d.heads * p.AB;
  int n_arg = 0;
  for (int a = 0; a < EGC_MAX_AGGR; ++a) {
    p.aggr[a] = a < d.n_aggr ? d.aggr[a] : -1;
    p.arg_slot[a] = (a < d.n_aggr && (d.aggr[a] == EGC_AGGR_MAX || d.aggr[a] == EGC_AGGR_MIN)) ? n_arg++ : -1;
  }
  p.n_arg = n_arg;
  p.n_saved = n_saved_slots(d);
  p.sigmoid = d.sigmoid;
  p.relu = d.relu;
  const int vec = vec4 ? 4 : 1;
  p.nvec = (p.BD + vec - 1) / vec;
  int g = 1;
  while (g < 32 && g < p.nvec) g <<= 1;
  p.G = g;
  p.n_pass = p.nvec > 32 ? (p.nvec + 31) / 32 : 1;
  auto a4 = [](int v) { return (v + 3) & ~3; };
  int off = 0;
  p.sm_agg = off; off = a4(off + p.A * p.BD);
  p.sm_w = off; off = a4(off + p.HAB);
  p.sm_per_warp = off;
  return off * kAggWarps * static_cast<int>(sizeof(float));
}

static int validate_desc(const egc_layer_desc* d, const char* who) {
  EGC_REQUIRE(d != nullptr, "%s: null descriptor", who);
  EGC_REQUIRE(d->n_dst > 0 && d->n_src > 0, "%s: n_dst=%d n_src=%d", who, d->n_dst, d->n_src);
  EGC_REQUIRE(d->heads > 0 && d->bases > 0 && d->dim > 0, "%s: heads=%d bases=%d dim=%d", who, d->heads, d->bases, d->dim);
  EGC_REQUIRE(d->n_aggr >= 1 && d->n_aggr <= EGC_MAX_AGGR, "%s: n_aggr=%d", who, d->n_aggr);
  for (int a = 0; a < d->n_aggr; ++a)
    EGC_REQUIRE(d->aggr[a] >= EGC_AGGR_SUM && d->aggr[a] <= EGC_AGGR_STD, "%s: unknown aggregator code %d", who, d->aggr[a]);
  return EGC_OK;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

static void set_plan(AggParams& p, const egc_row_plan* plan) {
  p.n_long = plan ? plan->n_long : 0;
  p.n_chunks = plan ? plan->n_chunks : 0;
  p.long_rows = plan ? plan->long_rows : nullptr;
  p.long_chunk_ptr = plan ? plan->long_chunk_ptr : nullptr;
  p.chunk_row = plan ? plan->chunk_row : nullptr;
  p.chunk_begin = plan ? plan->chunk_begin : nullptr;
}

static int validate_plan(const egc_row_plan* plan, const char* who) {
  if (plan == nullptr || plan->n_long == 0) return EGC_OK;
  EGC_REQUIRE(plan->n_long > 0 && plan->n_chunks >= 2 * plan->n_long, "%s: inconsistent row plan", who);
  EGC_REQUIRE(plan->long_rows && plan->long_chunk_ptr && plan->chunk_row && plan->chunk_begin, "%s: row plan with null arrays", who);
  return EGC_OK;
}

// egc_dropout -> p.drop_*: threshold and scale from the fp32 p widened to double (include/egc_b200.h)
static int set_dropout(AggParams& p, const egc_layer_desc& d, const egc_epilogue* epi, const egc_dropout* dropout,
                       const float* out, const char* who) {
  p.drop_seed = nullptr;
  if (dropout == nullptr || dropout->p == 0.f) return EGC_OK;
  EGC_REQUIRE(dropout->p > 0.f && dropout->p < 1.f, "%s: dropout p=%g outside [0, 1)", who, static_cast<double>(dropout->p));
  EGC_REQUIRE(dropout->seed != nullptr, "%s: dropout without a seed", who);
  EGC_REQUIRE(d.relu != 0, "%s: dropout is fused after the ReLU: it needs desc->relu", who);
  EGC_REQUIRE(out != nullptr, "%s: dropout applies to the `out` output, which is not requested", who);
  EGC_REQUIRE(epi == nullptr || (epi->scale == nullptr && epi->shift == nullptr && epi->add == nullptr),
              "%s: dropout cannot be combined with the epilogue's scale / shift / add", who);
  EGC_REQUIRE(dropout->row_offset >= 0 && dropout->row_offset + d.n_dst <= (int64_t{1} << 32),
              "%s: dropout row_offset=%lld outside [0, 2^32 - n_dst]", who, static_cast<long long>(dropout->row_offset));
  const double keep = 1.0 - static_cast<double>(dropout->p);
  p.drop_seed = dropout->seed;
  p.drop_thresh = static_cast<uint32_t>(std::min(std::floor(keep * 4294967296.0), 4294967295.0));   // p < 2^-53: 1 - p == 1
  p.drop_scale = static_cast<float>(1.0 / keep);
  p.drop_row0 = dropout->row_offset;
  return EGC_OK;
}

}  // namespace egc

#include "backward_pass1.cuh"
#include "backward_pass2.cuh"
#include "backward_pass2_ring.cuh"
#include "backward_route.cuh"

namespace egc {

constexpr int kBf16RingDepth = 8;

// which target-side streams does this aggregator list need?  bit0 sym, bit1 lin, bit2 sq
static int stream_mask_of(const egc_layer_desc& d, bool& has_route) {
  int m = 0;
  has_route = false;
  for (int a = 0; a < d.n_aggr; ++a) {
    switch (d.aggr[a]) {
      case EGC_AGGR_SUM: case EGC_AGGR_MEAN: m |= 2; break;
      case EGC_AGGR_SYMNORM: m |= 1; break;
      case EGC_AGGR_VAR: case EGC_AGGR_STD: m |= 2 | 4; break;
      case EGC_AGGR_MAX: case EGC_AGGR_MIN: has_route = true; break;
    }
  }
  return m;
}

static int combine_bwd_grid(int n_rows) { return std::max(1, std::min(ceil_div(n_rows, kAggWarps), sm_count() * 4)); }

struct BwdLayout {
  size_t ts_bytes, csc_part_bytes, colsum_bytes, route_bytes, total;
  int n_ts, ts_sym, ts_lin, ts_sq, tsmask;
  bool has_route;
};

// ts_elem: bytes per stored target-side stream value (4, or 2 with bf16 storage)
static BwdLayout bwd_layout(const egc_layer_desc& d, const egc_row_plan* csc_plan, size_t ts_elem = 4) {
  BwdLayout L{};
  L.tsmask = stream_mask_of(d, L.has_route);
  int s = 0;
  L.ts_sym = (L.tsmask & 1) ? s++ : -1;
  L.ts_lin = (L.tsmask & 2) ? s++ : -1;
  L.ts_sq = (L.tsmask & 4) ? s++ : -1;
  L.n_ts = s;
  const size_t bd = static_cast<size_t>(d.bases) * d.dim;
  L.ts_bytes = align_up(static_cast<size_t>(d.n_dst) * std::max(L.n_ts, 1) * bd * ts_elem, 256);
  L.csc_part_bytes = align_up(static_cast<size_t>(csc_plan ? csc_plan->n_chunks : 0) * std::max(L.n_ts, 1) * bd * 4, 256) +
                     align_up(static_cast<size_t>(csc_plan ? csc_plan->n_long : 0) * sizeof(int), 256) +
                     256;   // + the task counter of k_scatter_cols
  // per-CTA column-sum partials of the fused pass-1 kernel, or the two-stage colsum scratch when it cannot fuse
  const size_t hd = static_cast<size_t>(d.heads) * d.dim, hab = static_cast<size_t>(d.heads) * d.n_aggr * d.bases;
  const size_t fused = static_cast<size_t>(combine_bwd_grid(d.n_dst)) * (hd + hab) * sizeof(float) + 256;
  L.colsum_bytes = align_up(std::max(fused, std::max(colsum_workspace_bytes(d.n_dst, static_cast<int>(hd)),
                                                     colsum_workspace_bytes(d.n_dst, static_cast<int>(hab)))), 256);
  L.route_bytes = align_up(static_cast<size_t>(d.n_dst) * n_arg_slots(d) * bd * 4, 256);
  L.total = L.ts_bytes + L.csc_part_bytes + L.colsum_bytes + L.route_bytes + 256;
  return L;
}

// Pass 2 of the backward: per source column over a CSC view, atomic-free.  d_bases[j] (= | +=) the column's sum of
// val_sym t_sym[i] + val_lin (t_lin[i] + 2 bases[j] t_sq[i]) over its entries; `csc_part` = chunk partials, the long-column
// counters and the task counter (BwdLayout::csc_part_bytes).
static int run_pass2(const egc_layer_desc& desc, const BwdLayout& L, const int32_t* colptr, const int32_t* rowidx,
                     const float* csc_val_sym, const float* csc_val_lin, const egc_row_plan* csc_plan, const float* tstreams,
                     const float* bases, float* d_bases, int col_begin, int col_end, bool accumulate, float* csc_part, bool vec4,
                     cudaStream_t st, bool bf16_store = false) {
  const int bd = desc.bases * desc.dim;
  AggParams geo{};
  fill_agg_params(geo, desc, vec4);
  ScatterParams s{};
  s.colptr = colptr; s.rowidx = rowidx; s.val_sym = csc_val_sym; s.val_lin = csc_val_lin; s.n_cols = desc.n_src;
  s.col_begin = col_begin;
  s.col_end = col_end;
  s.n_long = csc_plan ? csc_plan->n_long : 0;
  s.n_chunks = csc_plan ? csc_plan->n_chunks : 0;
  s.long_rows = csc_plan ? csc_plan->long_rows : nullptr;
  s.long_chunk_ptr = csc_plan ? csc_plan->long_chunk_ptr : nullptr;
  s.chunk_row = csc_plan ? csc_plan->chunk_row : nullptr;
  s.chunk_begin = csc_plan ? csc_plan->chunk_begin : nullptr;
  s.partials = csc_part;
  const size_t part_bytes = align_up(static_cast<size_t>(s.n_chunks) * std::max(L.n_ts, 1) * bd * 4, 256);
  const size_t counters_bytes = align_up(static_cast<size_t>(s.n_long) * sizeof(int), 256);
  int* long_counter = reinterpret_cast<int*>(reinterpret_cast<char*>(csc_part) + part_bytes);
  int* task_counter = reinterpret_cast<int*>(reinterpret_cast<char*>(long_counter) + counters_bytes);
  // column-block kernel: 128-bit pieces, unweighted entries, one pass, interleaved streams
  // (EGC_BWD_WARP_PER_COLUMN=1 keeps the warp-per-column kernel)
  static const bool legacy_cols = getenv("EGC_BWD_WARP_PER_COLUMN") != nullptr;
  const bool col_blocks = vec4 && csc_val_lin == nullptr && geo.n_pass == 1 && (geo.G == 32 || geo.G == 16) && (!legacy_cols || bf16_store);
  EGC_REQUIRE(col_blocks || !bf16_store, "egc_aggregate_bwd_bf16: the column pass needs rows of 36..128 values, a multiple of 4, 16-byte "
              "aligned, and no per-entry linear weights");
  const bool fuse_merge = geo.n_pass == 1 && s.n_long > 0;     // the last chunk warp of a long column merges its partials
  s.long_counter = (col_blocks || fuse_merge) ? long_counter : nullptr;
  s.tstreams = tstreams; s.bases = bases; s.d_bases = d_bases;
  s.n_ts = L.n_ts; s.ts_sym = L.ts_sym; s.ts_lin = L.ts_lin; s.ts_sq = L.ts_sq;
  s.BD = bd; s.nvec = geo.nvec; s.G = geo.G; s.n_pass = geo.n_pass;
  s.ts_row_stride = static_cast<int64_t>(L.n_ts) * bd;
  s.off_sym = L.ts_sym < 0 ? 0 : static_cast<int64_t>(L.ts_sym) * bd;
  s.off_lin = L.ts_lin < 0 ? 0 : static_cast<int64_t>(L.ts_lin) * bd;
  s.off_sq = L.ts_sq < 0 ? 0 : static_cast<int64_t>(L.ts_sq) * bd;
  s.routed = accumulate ? 1 : 0;
  // L2 locality hints of the column-block kernel: target rows whose streams lie within a 64 MB span around the column id
  // are fetched evict_last, the rest evict_first.  Measured on B200 (profiles/r02o_l2_hints.txt): arxiv-shaped EGC-M
  // (three streams, 1536 B per target) 0.376 -> 0.332 ms, no change on the uniform graph; mag-shaped EGC-S (one stream,
  // 256 B per target) 0.289 -> 0.362 ms - so the default is on for layers with two or more streams only.
  // EGC_BWD_NEAR_MB overrides the span for every layer (0 = no hints).
  static const int near_env = [] { const char* e = getenv("EGC_BWD_NEAR_MB"); return e ? std::max(0, atoi(e)) : -1; }();
  const int near_mb = near_env >= 0 ? near_env : (L.n_ts >= 2 ? 64 : 0);
  const int64_t ts_elem = bf16_store ? 2 : 4;
  s.near_rows = static_cast<int>(std::min<int64_t>(int64_t{1} << 30, (static_cast<int64_t>(near_mb) << 20) /
                                                       std::max<int64_t>(1, static_cast<int64_t>(std::max(L.n_ts, 1)) * bd * ts_elem * 2)));
  s.mode = 0;
  if (s.col_end <= s.col_begin) return EGC_OK;
  if (col_blocks) {
    EGC_CUDA(cudaMemsetAsync(long_counter, 0, counters_bytes + sizeof(int), st));
    // ring variant (rows land in a per-warp shared-memory ring, R entries ahead across columns): 128-float rows, two or more
    // streams.  Measured on B200, arxiv-shaped EGC-M (profiles/r02r_ring.txt): 0.334 -> 0.282 ms (depth 4 = depth 7), uniform
    // graph 0.480 -> 0.439 ms.  EGC_BWD_RING = ring depth (4: three CTAs per SM, 7: two), 0 = the register-gather kernel.
    static const int ring = [] { const char* e = getenv("EGC_BWD_RING"); return e ? atoi(e) : -1; }();
    if (bf16_store) {
      // bf16 streams: a slot holds half the bytes, so depth 8 keeps the fp32 ring's shared memory (and bytes in flight) per
      // warp at three CTAs per SM.  EGC_BWD_RING=4 selects the shallower ring, 0 the register-gather kernel.
      const int r = ring < 0 ? kBf16RingDepth : ring;
      if (r > 0 && geo.G == 32 && L.n_ts >= 2)
        return r >= 8 ? launch_scatter_ring<8, bf16>(s, L.tsmask, task_counter, st) : launch_scatter_ring<4, bf16>(s, L.tsmask, task_counter, st);
      return geo.G == 32 ? launch_scatter_cols<32, bf16>(s, L.tsmask, task_counter, st) : launch_scatter_cols<16, bf16>(s, L.tsmask, task_counter, st);
    }
    const int r = ring < 0 ? 4 : ring;
    if (r > 0 && geo.G == 32 && L.n_ts >= 2)
      return r >= 7 ? launch_scatter_ring<7>(s, L.tsmask, task_counter, st) : launch_scatter_ring<4>(s, L.tsmask, task_counter, st);
    return geo.G == 32 ? launch_scatter_cols<32>(s, L.tsmask, task_counter, st) : launch_scatter_cols<16>(s, L.tsmask, task_counter, st);
  }
  if (fuse_merge) EGC_CUDA(cudaMemsetAsync(long_counter, 0, counters_bytes, st));
  if (int rc = launch_scatter(s, L.tsmask, vec4, csc_val_lin != nullptr, st)) return rc;
  if (s.n_long > 0 && !fuse_merge) {
    s.mode = 1;
    if (int rc = launch_scatter(s, L.tsmask, vec4, csc_val_lin != nullptr, st)) return rc;
  }
  return EGC_OK;
}

}  // namespace egc

using namespace egc;

extern "C" {

int32_t egc_saved_slots(const egc_layer_desc* desc) { return desc ? n_saved_slots(*desc) : 0; }
int32_t egc_saved_arg_slots(const egc_layer_desc* desc) { return desc ? n_arg_slots(*desc) : 0; }

size_t egc_aggregate_fwd_workspace_bytes(const egc_layer_desc* desc, const egc_row_plan* plan) {
  if (desc == nullptr) return 0;
  const int mask = prim_mask_of(*desc);
  if (mask <= 0) return 0;
  const size_t bd = static_cast<size_t>(desc->bases) * desc->dim;
  return align_up(static_cast<size_t>(plan ? plan->n_chunks : 0) * n_slots_of_mask(mask) * bd * 4, 256) +
         align_up(static_cast<size_t>(plan ? plan->n_long : 0) * sizeof(int), 256) + 256;
}

int egc_aggregate_fwd(const egc_layer_desc* desc, const int32_t* rowptr, const int32_t* col, const float* val_sym,
                      const float* val_lin, const egc_row_plan* plan, const float* bases, const float* weightings,
                      const float* bias, const egc_epilogue* epilogue, const int32_t* row_subset, int32_t n_subset, float* out, float* agg_out,
                      int32_t* arg_out, float* saved, int32_t* saved_arg, void* workspace, size_t workspace_bytes,
                      void* stream) {
  return egc_aggregate_fwd_dropout(desc, rowptr, col, val_sym, val_lin, plan, bases, weightings, bias, epilogue, nullptr,
                                   row_subset, n_subset, out, agg_out, arg_out, saved, saved_arg, workspace, workspace_bytes,
                                   stream);
}

int egc_aggregate_fwd_dropout(const egc_layer_desc* desc, const int32_t* rowptr, const int32_t* col, const float* val_sym,
                              const float* val_lin, const egc_row_plan* plan, const float* bases, const float* weightings,
                              const float* bias, const egc_epilogue* epilogue, const egc_dropout* dropout,
                              const int32_t* row_subset, int32_t n_subset, float* out, float* agg_out, int32_t* arg_out,
                              float* saved, int32_t* saved_arg, void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = validate_desc(desc, "egc_aggregate_fwd")) return rc;
  if (int rc = validate_plan(plan, "egc_aggregate_fwd")) return rc;
  EGC_REQUIRE(rowptr && col && bases, "egc_aggregate_fwd: null graph / bases pointer");
  EGC_REQUIRE(out == nullptr || weightings != nullptr, "egc_aggregate_fwd: weightings required to produce out");
  EGC_REQUIRE(out || agg_out || arg_out || saved, "egc_aggregate_fwd: no output requested");
  EGC_REQUIRE(n_subset >= 0 && (n_subset == 0 || row_subset != nullptr), "egc_aggregate_fwd: bad row subset");
  const int mask = prim_mask_of(*desc);
  EGC_REQUIRE(!(mask & P_SYM) || val_sym != nullptr, "egc_aggregate_fwd: symnorm requested without val_sym");
  EGC_REQUIRE(!((mask & P_SYM) && val_lin), "egc_aggregate_fwd: val_lin cannot be combined with symnorm (ref :253-254)");
  EGC_REQUIRE(workspace_bytes >= egc_aggregate_fwd_workspace_bytes(desc, plan) && (workspace || !(plan && plan->n_chunks)),
              "egc_aggregate_fwd: workspace too small");
  const int n_arg = n_arg_slots(*desc);
  EGC_REQUIRE(saved == nullptr || n_arg == 0 || saved_arg != nullptr, "egc_aggregate_fwd: saved_arg required with saved for min/max");
  AggParams p{};
  const int bd = desc->bases * desc->dim;
  const bool vec4 = (bd % 4 == 0) && aligned16(bases) && aligned16(out) && aligned16(agg_out) && aligned16(workspace) &&
                    aligned16(arg_out) && aligned16(saved) && aligned16(saved_arg);
  const int smem = fill_agg_params(p, *desc, vec4);
  EGC_REQUIRE(smem <= 200 * 1024, "egc_aggregate_fwd: layer too wide for the shared-memory staging (%d bytes)", smem);
  p.rowptr = rowptr; p.col = col; p.val_sym = val_sym; p.val_lin = val_lin; p.n_rows = desc->n_dst;
  p.row_map = row_subset;
  p.n_row_tasks = row_subset != nullptr ? n_subset : desc->n_dst;
  set_plan(p, plan);
  p.partials = static_cast<float*>(workspace);
  p.n_slots = n_slots_of_mask(mask);
  p.long_counter = reinterpret_cast<int*>(static_cast<char*>(workspace) +
                                          align_up(static_cast<size_t>(p.n_chunks) * p.n_slots * bd * 4, 256));
  p.bases = bases; p.weightings = weightings; p.bias = bias;
  if (epilogue != nullptr) {
    EGC_REQUIRE((epilogue->scale == nullptr) == (epilogue->shift == nullptr), "egc_aggregate_fwd: epilogue scale and shift come together");
    EGC_REQUIRE(out != nullptr || (!epilogue->scale && !epilogue->add), "egc_aggregate_fwd: an epilogue needs the `out` output");
    p.epi_scale = epilogue->scale; p.epi_shift = epilogue->shift; p.epi_add = epilogue->add;
    if (epilogue->agg_init != nullptr) {
      for (int a = 0; a < desc->n_aggr; ++a)
        EGC_REQUIRE(desc->aggr[a] == EGC_AGGR_SUM || desc->aggr[a] == EGC_AGGR_SYMNORM,
                    "egc_aggregate_fwd: agg_init continues sums - every aggregator must be sum or symnorm");
      EGC_REQUIRE(aligned16(epilogue->agg_init), "egc_aggregate_fwd: agg_init must be 16-byte aligned");
      p.agg_init = epilogue->agg_init;
    }
  }
  if (int rc = set_dropout(p, *desc, epilogue, dropout, out, "egc_aggregate_fwd")) return rc;
  p.out = out; p.agg_out = agg_out; p.arg_out = arg_out; p.saved = saved; p.saved_arg = saved_arg;
  cudaStream_t st = as_stream(stream);
  const bool want_arg = (arg_out != nullptr || saved_arg != nullptr) && n_arg > 0;
  if (arg_out != nullptr && !want_arg && row_subset == nullptr)   // no min/max slot: every arg is "none"
    EGC_CUDA(cudaMemsetAsync(arg_out, 0xff, static_cast<size_t>(desc->n_dst) * desc->n_aggr * bd * sizeof(int32_t), st));
  // dropout runs the DROP = true instantiations (*_dropout.cu); every other call the kernels without dropout code
  const bool drop = p.drop_seed != nullptr;
  auto launch = drop ? (vec4 ? launch_aggregate_v4_dropout : launch_aggregate_v1_dropout)
                     : (vec4 ? launch_aggregate_v4 : launch_aggregate_v1);
  p.mode = 0;
  const int hd = desc->heads * desc->dim;
  // (agg_init - the opt-in split launches of a row-partitioned caller - is served by the general kernel only)
  const bool fast = vec4 && val_lin == nullptr && p.agg_init == nullptr && p.n_pass == 1 && (p.G == 32 || p.G == 16) &&
                    hd <= ((desc->dim % 4 == 0) ? 512 : 128) && static_cast<int64_t>(desc->n_src) * bd < (int64_t{1} << 32) &&
                    (desc->dim % 4 != 0 || (aligned16(bias) && aligned16(p.epi_scale) && aligned16(p.epi_shift) && aligned16(p.epi_add)));
  const int static_idx = fast ? static_cfg_index(*desc) : -1;
  // row-block kernel: whole-graph calls of the specialised shapes (EGC_FWD_WARP_PER_ROW=1 keeps the warp-per-row kernel)
  static const bool legacy_rows = getenv("EGC_FWD_WARP_PER_ROW") != nullptr;
  // needs the window + 8 rows of weights per warp in shared memory (3 CTAs per SM)
  const bool row_blocks = fast && !legacy_rows && rows_kernel_smem_bytes(p) <= 72 * 1024;
  const size_t counter_off = align_up(static_cast<size_t>(p.n_long) * sizeof(int), 256);   // inside the trailing 256 B
  int* task_counter = reinterpret_cast<int*>(reinterpret_cast<char*>(p.long_counter) + counter_off);
  if (row_blocks) EGC_CUDA(cudaMemsetAsync(p.long_counter, 0, counter_off + sizeof(int), st));
  else if (fast && p.n_long > 0) EGC_CUDA(cudaMemsetAsync(p.long_counter, 0, static_cast<size_t>(p.n_long) * sizeof(int), st));
  if (row_blocks && static_idx >= 0) {
    if (int rc = (drop ? launch_aggregate_rows_static_dropout : launch_aggregate_rows_static)(static_idx, p, want_arg, task_counter, st)) return rc;
  } else if (row_blocks) {
    auto rows = drop ? (p.G == 32 ? launch_aggregate_rows_g32_dropout : launch_aggregate_rows_g16_dropout)
                     : (p.G == 32 ? launch_aggregate_rows_g32 : launch_aggregate_rows_g16);
    if (int rc = rows(p, mask, want_arg, task_counter, st)) return rc;
  } else if (static_idx >= 0) {
    if (int rc = (drop ? launch_aggregate_fast_static_dropout : launch_aggregate_fast_static)(static_idx, p, want_arg, smem, st)) return rc;
  } else if (fast) {
    auto fast_fam = drop ? (p.G == 32 ? launch_aggregate_fast_g32_dropout : launch_aggregate_fast_g16_dropout)
                         : (p.G == 32 ? launch_aggregate_fast_g32 : launch_aggregate_fast_g16);
    if (int rc = fast_fam(p, mask, want_arg, smem, st)) return rc;
  } else {
    if (int rc = launch(p, mask, val_lin != nullptr, want_arg, smem, st)) return rc;
  }
  if (p.n_long > 0 && !fast) {                  // the fast kernels merge long rows themselves
    p.mode = 1;
    if (int rc = launch(p, mask, val_lin != nullptr, want_arg, smem, st)) return rc;
  }
  return EGC_OK;
}

int egc_aggregate_fwd_bf16(const egc_layer_desc* desc, const int32_t* rowptr, const int32_t* col, const float* val_sym,
                           const egc_row_plan* plan, const uint16_t* bases, const float* weightings, const float* bias,
                           const egc_epilogue* epilogue, float* out, float* agg_out, int32_t* arg_out, float* saved,
                           int32_t* saved_arg, void* workspace, size_t workspace_bytes, void* stream) {
  return egc_aggregate_fwd_bf16_dropout(desc, rowptr, col, val_sym, plan, bases, weightings, bias, epilogue, nullptr, out,
                                        agg_out, arg_out, saved, saved_arg, workspace, workspace_bytes, stream);
}

int egc_aggregate_fwd_bf16_dropout(const egc_layer_desc* desc, const int32_t* rowptr, const int32_t* col, const float* val_sym,
                                   const egc_row_plan* plan, const uint16_t* bases, const float* weightings, const float* bias,
                                   const egc_epilogue* epilogue, const egc_dropout* dropout, float* out, float* agg_out,
                                   int32_t* arg_out, float* saved, int32_t* saved_arg, void* workspace, size_t workspace_bytes,
                                   void* stream) {
  if (int rc = validate_desc(desc, "egc_aggregate_fwd_bf16")) return rc;
  if (int rc = validate_plan(plan, "egc_aggregate_fwd_bf16")) return rc;
  EGC_REQUIRE(rowptr && col && bases, "egc_aggregate_fwd_bf16: null graph / bases pointer");
  EGC_REQUIRE(out == nullptr || weightings != nullptr, "egc_aggregate_fwd_bf16: weightings required to produce out");
  EGC_REQUIRE(out || agg_out || arg_out || saved, "egc_aggregate_fwd_bf16: no output requested");
  const int mask = prim_mask_of(*desc);
  EGC_REQUIRE(!(mask & P_SYM) || val_sym != nullptr, "egc_aggregate_fwd_bf16: symnorm requested without val_sym");
  EGC_REQUIRE(workspace_bytes >= egc_aggregate_fwd_workspace_bytes(desc, plan) && workspace != nullptr,
              "egc_aggregate_fwd_bf16: workspace too small");
  const int n_arg = n_arg_slots(*desc);
  EGC_REQUIRE(saved == nullptr || n_arg == 0 || saved_arg != nullptr, "egc_aggregate_fwd_bf16: saved_arg required with saved for min/max");
  const int bd = desc->bases * desc->dim, hd = desc->heads * desc->dim;
  EGC_REQUIRE(bd % 8 == 0 && bd >= 40 && bd <= 128,
              "egc_aggregate_fwd_bf16: bf16 storage covers basis rows of 40..128 values, a multiple of 8 (B*D = %d)", bd);
  EGC_REQUIRE(aligned16(bases) && aligned16(out) && aligned16(agg_out) && aligned16(workspace) && aligned16(arg_out) &&
              aligned16(saved) && aligned16(saved_arg), "egc_aggregate_fwd_bf16: tensors must be 16-byte aligned");
  EGC_REQUIRE(hd <= ((desc->dim % 4 == 0) ? 512 : 128), "egc_aggregate_fwd_bf16: H*D = %d outputs per row exceed one pass", hd);
  EGC_REQUIRE(static_cast<int64_t>(desc->n_src) * bd < (int64_t{1} << 32), "egc_aggregate_fwd_bf16: bases exceed 2^32 values");
  AggParams p{};
  fill_agg_params(p, *desc, true);
  p.nvec = bd / 8;                                     // 16-byte pieces of 8 bf16 values
  p.G = p.nvec > 8 ? 16 : 8;
  p.n_pass = 1;
  EGC_REQUIRE(rows_kernel_smem_bytes(p) <= 72 * 1024, "egc_aggregate_fwd_bf16: layer too wide for the row-block staging (%d bytes)",
              rows_kernel_smem_bytes(p));
  p.rowptr = rowptr; p.col = col; p.val_sym = val_sym; p.val_lin = nullptr; p.n_rows = desc->n_dst;
  p.row_map = nullptr;
  p.n_row_tasks = desc->n_dst;
  set_plan(p, plan);
  p.partials = static_cast<float*>(workspace);
  p.n_slots = n_slots_of_mask(mask);
  p.long_counter = reinterpret_cast<int*>(static_cast<char*>(workspace) +
                                          align_up(static_cast<size_t>(p.n_chunks) * p.n_slots * bd * 4, 256));
  p.bases = reinterpret_cast<const float*>(bases);     // bf16 rows (k_aggregate_rows<.., bf16> reads them as such)
  p.weightings = weightings; p.bias = bias;
  if (epilogue != nullptr) {
    EGC_REQUIRE((epilogue->scale == nullptr) == (epilogue->shift == nullptr), "egc_aggregate_fwd_bf16: epilogue scale and shift come together");
    EGC_REQUIRE(out != nullptr || (!epilogue->scale && !epilogue->add), "egc_aggregate_fwd_bf16: an epilogue needs the `out` output");
    EGC_REQUIRE(epilogue->agg_init == nullptr, "egc_aggregate_fwd_bf16: agg_init is not supported");
    p.epi_scale = epilogue->scale; p.epi_shift = epilogue->shift; p.epi_add = epilogue->add;
  }
  EGC_REQUIRE(desc->dim % 4 != 0 || (aligned16(bias) && aligned16(p.epi_scale) && aligned16(p.epi_shift) && aligned16(p.epi_add)),
              "egc_aggregate_fwd_bf16: bias / epilogue tensors must be 16-byte aligned");
  if (int rc = set_dropout(p, *desc, epilogue, dropout, out, "egc_aggregate_fwd_bf16")) return rc;
  p.out = out; p.agg_out = agg_out; p.arg_out = arg_out; p.saved = saved; p.saved_arg = saved_arg;
  cudaStream_t st = as_stream(stream);
  const bool want_arg = (arg_out != nullptr || saved_arg != nullptr) && n_arg > 0;
  if (arg_out != nullptr && !want_arg)                 // no min/max slot: every arg is "none"
    EGC_CUDA(cudaMemsetAsync(arg_out, 0xff, static_cast<size_t>(desc->n_dst) * desc->n_aggr * bd * sizeof(int32_t), st));
  p.mode = 0;
  const size_t counter_off = align_up(static_cast<size_t>(p.n_long) * sizeof(int), 256);
  int* task_counter = reinterpret_cast<int*>(reinterpret_cast<char*>(p.long_counter) + counter_off);
  EGC_CUDA(cudaMemsetAsync(p.long_counter, 0, counter_off + sizeof(int), st));
  const int static_idx = static_cfg_index(*desc);
  if (p.drop_seed != nullptr) {                       // the DROP = true instantiations (*_dropout.cu)
    if (static_idx >= 0) return launch_aggregate_rows_bf16_static_dropout(static_idx, p, want_arg, task_counter, st);
    return (p.G == 16 ? launch_aggregate_rows_bf16_g16_dropout : launch_aggregate_rows_bf16_g8_dropout)(p, mask, want_arg, task_counter, st);
  }
  if (static_idx >= 0) return launch_aggregate_rows_bf16_static(static_idx, p, want_arg, task_counter, st);
  return (p.G == 16 ? launch_aggregate_rows_bf16_g16 : launch_aggregate_rows_bf16_g8)(p, mask, want_arg, task_counter, st);
}

size_t egc_aggregate_bwd_workspace_bytes(const egc_layer_desc* desc, const egc_row_plan* csc_plan, int32_t flags) {
  (void)flags;
  if (desc == nullptr || prim_mask_of(*desc) <= 0) return 0;
  return bwd_layout(*desc, csc_plan).total;
}

}  // extern "C"

// egc_aggregate_bwd / egc_aggregate_bwd_bf16.  bf16: `bases` points at bf16 rows and the target-side streams are stored as
// bf16 in the workspace (bwd_layout with 2-byte elements); every other tensor and all arithmetic stay fp32.
static int aggregate_bwd_impl(const egc_layer_desc* desc, const int32_t* rowptr, const int32_t* col, const float* val_lin,
                              const int32_t* colptr, const int32_t* rowidx, const int32_t* csr2csc, const float* csc_val_sym,
                              const float* csc_val_lin, const egc_row_plan* csc_plan, const float* bases,
                              const float* weightings, const float* saved, const int32_t* saved_arg, const float* grad_out,
                              const float* out_act, const float* epi_scale, float* d_weightings, float* d_bases, float* d_bias,
                              float* d_lin_colsum, float* tstreams_out, int32_t flags, int32_t col_split, void* workspace,
                              size_t workspace_bytes, void* stream, bool bf16_store) {
  if (int rc = validate_desc(desc, "egc_aggregate_bwd")) return rc;
  if (int rc = validate_plan(csc_plan, "egc_aggregate_bwd")) return rc;
  const bool pass1_only = (flags & EGC_BWD_PASS1_ONLY) != 0;
  EGC_REQUIRE(!bf16_store || (val_lin == nullptr && csc_val_lin == nullptr),
              "egc_aggregate_bwd_bf16: no per-entry linear weights");
  EGC_REQUIRE(rowptr && col && bases && weightings && saved && grad_out && d_weightings && workspace &&
              (pass1_only || (colptr && rowidx && d_bases)), "egc_aggregate_bwd: null pointer");
  EGC_REQUIRE((desc->relu != 0) == (out_act != nullptr), "egc_aggregate_bwd: out_act must be given exactly when desc->relu is set");
  const size_t ts_elem = bf16_store ? 2 : 4;
  const BwdLayout L = bwd_layout(*desc, csc_plan, ts_elem);
  const bool det_route = (flags & EGC_BWD_DETERMINISTIC) != 0 && L.has_route;
  EGC_REQUIRE(!det_route || csr2csc != nullptr, "egc_aggregate_bwd: EGC_BWD_DETERMINISTIC needs csr2csc");
  const int mask = prim_mask_of(*desc);
  const int n_arg = n_arg_slots(*desc);
  EGC_REQUIRE(n_arg == 0 || saved_arg != nullptr, "egc_aggregate_bwd: saved_arg required for min/max");
  EGC_REQUIRE(!(mask & P_SYM) || csc_val_sym || pass1_only, "egc_aggregate_bwd: symnorm requested without csc_val_sym");
  EGC_REQUIRE((val_lin == nullptr) == (csc_val_lin == nullptr), "egc_aggregate_bwd: val_lin and csc_val_lin must come together");
  EGC_REQUIRE(!((mask & P_SYM) && val_lin), "egc_aggregate_bwd: val_lin cannot be combined with symnorm");
  EGC_REQUIRE(workspace_bytes >= L.total, "egc_aggregate_bwd: workspace too small (%zu < %zu)", workspace_bytes, L.total);
  EGC_REQUIRE(L.ts_bytes / ts_elem < (size_t{1} << 32), "egc_aggregate_bwd: target-side streams exceed 2^32 values");
  // Column phases (row-partitioned callers): HEAD = pass 1, routing and pass 2 of the source columns >= col_split (the
  // halo columns, whose partial sums travel to their owners while ...) TAIL = pass 2 of the columns < col_split runs.
  const bool head = (flags & EGC_BWD_COLS_HEAD) != 0, tail = (flags & EGC_BWD_COLS_TAIL) != 0;
  EGC_REQUIRE(!(head && tail), "egc_aggregate_bwd: EGC_BWD_COLS_HEAD and EGC_BWD_COLS_TAIL are separate calls");
  const bool split = head || tail;
  EGC_REQUIRE(!pass1_only || (!split && !L.has_route && tstreams_out != nullptr),
              "egc_aggregate_bwd: EGC_BWD_PASS1_ONLY needs tstreams_out, a layer without min / max and no column phase");
  EGC_REQUIRE(aligned16(tstreams_out), "egc_aggregate_bwd: tstreams_out must be 16-byte aligned");
  EGC_REQUIRE(!split || (col_split >= 0 && col_split <= desc->n_src), "egc_aggregate_bwd: col_split=%d outside [0, %d]", col_split, desc->n_src);
  cudaStream_t st = as_stream(stream);
  char* ws = static_cast<char*>(workspace);
  float* tstreams = tstreams_out != nullptr ? tstreams_out : reinterpret_cast<float*>(ws);
  float* csc_part = reinterpret_cast<float*>(ws + L.ts_bytes);
  void* colsum_ws = ws + L.ts_bytes + L.csc_part_bytes;
  float* t_route = reinterpret_cast<float*>(ws + L.ts_bytes + L.csc_part_bytes + L.colsum_bytes);

  const int bd = desc->bases * desc->dim, hd = desc->heads * desc->dim;
  const int hab = desc->heads * desc->n_aggr * desc->bases;
  const bool vec4 = (bd % 4 == 0) && aligned16(bases) && aligned16(d_bases) && aligned16(workspace);
  const bool skip_route = (flags & EGC_BWD_SKIP_ROUTING) != 0;

  // Order of the routed min/max gradients and pass 2.  One call: pass 2 WRITES every row of d_bases (empty columns
  // included) and the routed gradients are added afterwards - no memset, no read-modify-write in pass 2.  Column phases:
  // the routing must be complete for the HEAD columns before the TAIL columns exist, so d_bases is zeroed, routed into,
  // and both pass-2 launches accumulate.  No linear stream at all (min / max only): zero + route, there is no pass 2.
  const bool route_first = split || L.tsmask == 0;
  if (!tail && route_first && (L.has_route || L.tsmask == 0))
    EGC_CUDA(cudaMemsetAsync(d_bases, 0, static_cast<size_t>(desc->n_src) * bd * sizeof(float), st));
  const bool pass2_accumulates = route_first && L.has_route;

  // ---- pass 1: streaming over target nodes
  bool fuse_colsum = false;
  if (!tail) {
    CombineBwdParams c{};
    c.rowptr = rowptr; c.col = col; c.val_lin = val_lin; c.n_rows = desc->n_dst;
    c.weightings = weightings; c.grad_out = grad_out; c.out_act = out_act; c.epi_scale = epi_scale; c.saved = saved; c.saved_arg = saved_arg;
    c.d_weightings = d_weightings; c.tstreams = tstreams; c.d_bases = d_bases;
    c.n_saved = n_saved_slots(*desc); c.n_arg = n_arg;
    c.n_ts = L.n_ts; c.ts_sym = L.ts_sym; c.ts_lin = L.ts_lin; c.ts_sq = L.ts_sq;
    c.H = desc->heads; c.B = desc->bases; c.D = desc->dim; c.A = desc->n_aggr;
    c.BD = bd; c.HD = hd; c.AB = desc->n_aggr * desc->bases; c.HAB = hab;
    int na = 0;
    for (int a = 0; a < EGC_MAX_AGGR; ++a) {
      c.aggr[a] = a < desc->n_aggr ? desc->aggr[a] : -1;
      c.arg_slot[a] = (a < desc->n_aggr && (desc->aggr[a] == EGC_AGGR_MAX || desc->aggr[a] == EGC_AGGR_MIN)) ? na++ : -1;
    }
    c.sigmoid = desc->sigmoid;
    auto a4 = [](int v) { return (v + 3) & ~3; };
    int off = 0;
    c.sm_w = off; off = a4(off + hab);
    c.sm_g = off; off = a4(off + hd);
    c.sm_saved = off; off = a4(off + c.n_saved * bd);
    c.sm_arg = off; off = a4(off + n_arg * bd);
    c.sm_per_warp = off;
    const int smem = (off * kAggWarps + 3 * hab) * static_cast<int>(sizeof(float));    // staging areas + index tables
    EGC_REQUIRE(smem <= 200 * 1024, "egc_aggregate_bwd: layer too wide for the shared-memory staging (%d bytes)", smem);
    c.ts_row_stride = static_cast<int64_t>(L.n_ts) * bd;       // interleaved: [n_dst][n_ts][BD]
    c.ts_stream_stride = bd;
    c.vec16 = (hab % 4 == 0 && hd % 4 == 0 && bd % 4 == 0 && aligned16(weightings) && aligned16(grad_out) &&
               aligned16(out_act) && aligned16(epi_scale) && aligned16(saved) && aligned16(saved_arg)) ? 1 : 0;
    const bool ev4 = (desc->dim % 4 == 0) && aligned16(tstreams);
    const bool linw = val_lin != nullptr;
    const int grid = combine_bwd_grid(desc->n_dst);
    // column sums fused into pass 1 when the per-lane accumulators cover the row widths
    fuse_colsum = (d_bias != nullptr || d_lin_colsum != nullptr) && hab <= 32 * kCbColIt &&
                  hd <= 32 * kCbColIt * (ev4 ? 4 : 1);
    c.colsum_part = fuse_colsum ? static_cast<float*>(colsum_ws) : nullptr;
    c.skip_route = skip_route ? 1 : 0;
    c.t_route = t_route;
#define EGC_LAUNCH_COMBINE_CFG(CFG, EV, LW, TS)                                                                \
    {                                                                                                          \
      auto kern = k_combine_bwd<CFG, EV, LW, TS>;                                                                \
      if (smem > 48 * 1024) EGC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
      LaunchScope egc_ls_("k_combine_bwd", st);                                                                \
      kern<<<grid, kAggThreads, smem, st>>>(c);                                                                \
    }
    using Dyn = DynCfg<0, 32>;
    const int static_idx = (ev4 && !linw && c.vec16) ? static_cfg_index(*desc) : -1;
    bool launched = false;
#define X(I, ...)                                                                                              \
    if (!launched && static_idx == I) {                                                                        \
      using SC = StaticCfg<__VA_ARGS__>;                                                                       \
      EGC_REQUIRE(SC::bsm_per_warp == c.sm_per_warp && SC::bsm_saved == c.sm_saved && SC::bsm_arg == c.sm_arg && \
                  SC::ts_sym == c.ts_sym && SC::ts_lin == c.ts_lin && SC::ts_sq == c.ts_sq,                    \
                  "egc_aggregate_bwd: static configuration %d disagrees with the host layout", I);             \
      if (bf16_store) EGC_LAUNCH_COMBINE_CFG(SC, 4, false, bf16)                                               \
      else EGC_LAUNCH_COMBINE_CFG(SC, 4, false, float)                                                                \
      launched = true;                                                                                         \
    }
    EGC_STATIC_CFGS(X)
#undef X
    if (launched) {
    } else if (bf16_store && ev4) EGC_LAUNCH_COMBINE_CFG(Dyn, 4, false, bf16)
    else if (bf16_store) EGC_LAUNCH_COMBINE_CFG(Dyn, 1, false, bf16)
    else if (ev4 && !linw) EGC_LAUNCH_COMBINE_CFG(Dyn, 4, false, float)
    else if (ev4 && linw) EGC_LAUNCH_COMBINE_CFG(Dyn, 4, true, float)
    else if (!linw) EGC_LAUNCH_COMBINE_CFG(Dyn, 1, false, float)
    else EGC_LAUNCH_COMBINE_CFG(Dyn, 1, true, float)
#undef EGC_LAUNCH_COMBINE_CFG
    EGC_LAUNCH_CHECK("k_combine_bwd");
    if (fuse_colsum) {
      {
        LaunchScope egc_ls_("k_colsum_partials", st);
        k_colsum_partials<<<ceil_div(hd + hab, 8), 256, 0, st>>>(c.colsum_part, grid, hd, hab, d_bias, d_lin_colsum);
      }
      EGC_LAUNCH_CHECK("k_colsum_partials");
    }
  }

  // ---- min/max routing: fp32 atomics in feature-slab order (default) or the CSC compare-and-add gather (deterministic)
  auto route = [&]() -> int {
    if (!L.has_route || skip_route) return EGC_OK;
    if (det_route) {
      const bool route_vec4 = vec4 && aligned16(saved_arg) && aligned16(t_route);
      AggParams geo{};
      fill_agg_params(geo, *desc, route_vec4);
      RouteCscParams r{};
      r.colptr = colptr; r.rowidx = rowidx; r.csr2csc = csr2csc; r.csc_val_lin = csc_val_lin; r.n_cols = desc->n_src;
      r.n_long = csc_plan ? csc_plan->n_long : 0;
      r.n_chunks = csc_plan ? csc_plan->n_chunks : 0;
      r.long_rows = csc_plan ? csc_plan->long_rows : nullptr;
      r.long_chunk_ptr = csc_plan ? csc_plan->long_chunk_ptr : nullptr;
      r.chunk_row = csc_plan ? csc_plan->chunk_row : nullptr;
      r.chunk_begin = csc_plan ? csc_plan->chunk_begin : nullptr;
      r.partials = csc_part;                     // not in use by pass 2 while the routing runs (stream order)
      r.saved_arg = saved_arg; r.t_route = t_route; r.d_bases = d_bases;
      r.n_arg = n_arg; r.BD = bd; r.nvec = geo.nvec; r.G = geo.G; r.n_pass = geo.n_pass;
      return launch_route_csc(r, route_vec4, st);
    }
    RouteParams r{};
    r.saved_arg = saved_arg; r.t_route = t_route; r.col = col; r.val_lin = val_lin; r.d_bases = d_bases;
    r.n_rows = desc->n_dst; r.n_arg = n_arg; r.BD = bd; r.n_slabs = ceil_div(bd, 32);
    // hubs = the long columns of the CSC plan (more than EGC_CHUNK_EDGES entries), privatised per CTA
    r.n_hubs = (csc_plan != nullptr && !(flags & EGC_BWD_NO_HUB_PRIVATISATION)) ? std::min(csc_plan->n_long, kRouteMaxHubs) : 0;
    r.hubs = r.n_hubs > 0 ? csc_plan->long_rows : nullptr;
    const int row_groups = ceil_div(desc->n_dst, kRouteRows);
    const int grid = std::max(1, std::min(ceil_div(row_groups, kRouteThreads / 32), sm_count()));
    const int smem = r.n_hubs > 0 ? 2 * kRouteHashSize * static_cast<int>(sizeof(int)) + r.n_hubs * 32 * static_cast<int>(sizeof(float)) : 0;
    if (smem > 48 * 1024) EGC_CUDA(cudaFuncSetAttribute(k_route_minmax, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    {
      LaunchScope egc_ls_("k_route_minmax", st);
      k_route_minmax<<<grid, kRouteThreads, smem, st>>>(r);
    }
    EGC_LAUNCH_CHECK("k_route_minmax");
    return EGC_OK;
  };
  if (!tail && route_first) {
    if (int rc = route()) return rc;
  }

  // ---- pass 2: per source column (CSC), atomic-free
  if (L.tsmask != 0 && !pass1_only) {
    if (int rc = run_pass2(*desc, L, colptr, rowidx, csc_val_sym, csc_val_lin, csc_plan, tstreams, bases, d_bases,
                           head ? col_split : 0, tail ? col_split : desc->n_src, pass2_accumulates, csc_part, vec4, st, bf16_store))
      return rc;
  }

  if (!tail && !route_first) {
    if (int rc = route()) return rc;
  }

  if (!tail && !fuse_colsum) {
    // a layer too wide for the fused column sums: with a fused epilogue, d_bias sums grad_out masked with out_act > 0 and
    // multiplied by epi_scale, the gradient pass 1 staged
    if (d_bias != nullptr) {
      if (int rc = colsum_f32(grad_out, desc->n_dst, hd, d_bias, colsum_ws, L.colsum_bytes, st, out_act, epi_scale)) return rc;
    }
    if (d_lin_colsum != nullptr) {
      if (int rc = colsum_f32(d_weightings, desc->n_dst, hab, d_lin_colsum, colsum_ws, L.colsum_bytes, st)) return rc;
    }
  }
  return EGC_OK;
}

extern "C" {

int egc_aggregate_bwd(const egc_layer_desc* desc, const int32_t* rowptr, const int32_t* col, const float* val_lin,
                      const int32_t* colptr, const int32_t* rowidx, const int32_t* csr2csc, const float* csc_val_sym,
                      const float* csc_val_lin, const egc_row_plan* csc_plan, const float* bases,
                      const float* weightings, const float* saved, const int32_t* saved_arg, const float* grad_out,
                      const float* out_act, const float* epi_scale, float* d_weightings, float* d_bases, float* d_bias,
                      float* d_lin_colsum, float* tstreams_out, int32_t flags, int32_t col_split, void* workspace,
                      size_t workspace_bytes, void* stream) {
  return aggregate_bwd_impl(desc, rowptr, col, val_lin, colptr, rowidx, csr2csc, csc_val_sym, csc_val_lin, csc_plan, bases,
                            weightings, saved, saved_arg, grad_out, out_act, epi_scale, d_weightings, d_bases, d_bias,
                            d_lin_colsum, tstreams_out, flags, col_split, workspace, workspace_bytes, stream, false);
}

size_t egc_aggregate_bwd_bf16_workspace_bytes(const egc_layer_desc* desc, const egc_row_plan* csc_plan, int32_t flags) {
  (void)flags;
  if (desc == nullptr || prim_mask_of(*desc) <= 0) return 0;
  return bwd_layout(*desc, csc_plan, 2).total;
}

int egc_aggregate_bwd_bf16(const egc_layer_desc* desc, const int32_t* rowptr, const int32_t* col, const int32_t* colptr,
                           const int32_t* rowidx, const int32_t* csr2csc, const float* csc_val_sym, const egc_row_plan* csc_plan,
                           const uint16_t* bases, const float* weightings, const float* saved, const int32_t* saved_arg,
                           const float* grad_out, const float* out_act, const float* epi_scale, float* d_weightings,
                           float* d_bases, float* d_bias, float* d_lin_colsum, int32_t flags, void* workspace,
                           size_t workspace_bytes, void* stream) {
  return egc_aggregate_bwd_bf16_partitioned(desc, rowptr, col, colptr, rowidx, csr2csc, csc_val_sym, csc_plan, bases, weightings,
                                            saved, saved_arg, grad_out, out_act, epi_scale, d_weightings, d_bases, d_bias,
                                            d_lin_colsum, nullptr, flags, 0, workspace, workspace_bytes, stream);
}

int egc_aggregate_bwd_bf16_partitioned(const egc_layer_desc* desc, const int32_t* rowptr, const int32_t* col,
                                       const int32_t* colptr, const int32_t* rowidx, const int32_t* csr2csc,
                                       const float* csc_val_sym, const egc_row_plan* csc_plan, const uint16_t* bases,
                                       const float* weightings, const float* saved, const int32_t* saved_arg,
                                       const float* grad_out, const float* out_act, const float* epi_scale, float* d_weightings,
                                       float* d_bases, float* d_bias, float* d_lin_colsum, uint16_t* tstreams_out,
                                       int32_t flags, int32_t col_split, void* workspace, size_t workspace_bytes, void* stream) {
  return aggregate_bwd_impl(desc, rowptr, col, nullptr, colptr, rowidx, csr2csc, csc_val_sym, nullptr, csc_plan,
                            reinterpret_cast<const float*>(bases), weightings, saved, saved_arg, grad_out, out_act, epi_scale,
                            d_weightings, d_bases, d_bias, d_lin_colsum, reinterpret_cast<float*>(tstreams_out), flags,
                            col_split, workspace, workspace_bytes, stream, true);
}

size_t egc_aggregate_bwd_cols_workspace_bytes(const egc_layer_desc* desc, const egc_row_plan* csc_plan) {
  if (desc == nullptr || prim_mask_of(*desc) <= 0) return 0;
  return bwd_layout(*desc, csc_plan).csc_part_bytes + 256;
}

}  // extern "C"

// egc_aggregate_bwd_cols / egc_aggregate_bwd_cols_bf16.  bf16: `tstreams` and `bases` point at bf16 rows; d_bases and the
// chunk partials in the workspace stay fp32, so both share egc_aggregate_bwd_cols_workspace_bytes().
static int aggregate_bwd_cols_impl(const egc_layer_desc* desc, const int32_t* colptr, const int32_t* rowidx,
                                   const float* csc_val_sym, const float* csc_val_lin, const egc_row_plan* csc_plan,
                                   const float* tstreams, const float* bases, float* d_bases, int32_t flags, void* workspace,
                                   size_t workspace_bytes, void* stream, bool bf16_store) {
  if (int rc = validate_desc(desc, "egc_aggregate_bwd_cols")) return rc;
  if (int rc = validate_plan(csc_plan, "egc_aggregate_bwd_cols")) return rc;
  EGC_REQUIRE(colptr && rowidx && tstreams && d_bases && workspace, "egc_aggregate_bwd_cols: null pointer");
  const size_t ts_elem = bf16_store ? 2 : 4;
  const BwdLayout L = bwd_layout(*desc, csc_plan, ts_elem);
  EGC_REQUIRE(!L.has_route, "egc_aggregate_bwd_cols: min / max gradients are routed by egc_aggregate_bwd, not by the column pass");
  EGC_REQUIRE(L.tsmask != 0, "egc_aggregate_bwd_cols: the layer has no linear stream");
  const int mask = prim_mask_of(*desc);
  EGC_REQUIRE(!(mask & P_SYM) || csc_val_sym, "egc_aggregate_bwd_cols: symnorm requested without csc_val_sym");
  EGC_REQUIRE(!((mask & P_SYM) && csc_val_lin), "egc_aggregate_bwd_cols: val_lin cannot be combined with symnorm");
  EGC_REQUIRE(L.ts_sq < 0 || bases != nullptr, "egc_aggregate_bwd_cols: var / std need the basis rows of the columns");
  EGC_REQUIRE(workspace_bytes >= L.csc_part_bytes, "egc_aggregate_bwd_cols: workspace too small (%zu < %zu)", workspace_bytes, L.csc_part_bytes);
  EGC_REQUIRE(L.ts_bytes / ts_elem < (size_t{1} << 32), "egc_aggregate_bwd_cols: target-side streams exceed 2^32 values");
  const int bd = desc->bases * desc->dim;
  const bool vec4 = (bd % 4 == 0) && (bases == nullptr || aligned16(bases)) && aligned16(d_bases) && aligned16(tstreams) && aligned16(workspace);
  return run_pass2(*desc, L, colptr, rowidx, csc_val_sym, csc_val_lin, csc_plan, tstreams, bases, d_bases, 0, desc->n_src,
                   (flags & EGC_BWD_ACCUMULATE) != 0, static_cast<float*>(workspace), vec4, as_stream(stream), bf16_store);
}

extern "C" {

int egc_aggregate_bwd_cols(const egc_layer_desc* desc, const int32_t* colptr, const int32_t* rowidx, const float* csc_val_sym,
                           const float* csc_val_lin, const egc_row_plan* csc_plan, const float* tstreams, const float* bases,
                           float* d_bases, int32_t flags, void* workspace, size_t workspace_bytes, void* stream) {
  return aggregate_bwd_cols_impl(desc, colptr, rowidx, csc_val_sym, csc_val_lin, csc_plan, tstreams, bases, d_bases, flags,
                                 workspace, workspace_bytes, stream, false);
}

int egc_aggregate_bwd_cols_bf16(const egc_layer_desc* desc, const int32_t* colptr, const int32_t* rowidx,
                                const float* csc_val_sym, const egc_row_plan* csc_plan, const uint16_t* tstreams,
                                const uint16_t* bases, float* d_bases, int32_t flags, void* workspace, size_t workspace_bytes,
                                void* stream) {
  return aggregate_bwd_cols_impl(desc, colptr, rowidx, csc_val_sym, nullptr, csc_plan, reinterpret_cast<const float*>(tstreams),
                                 reinterpret_cast<const float*>(bases), d_bases, flags, workspace, workspace_bytes, stream, true);
}

}  // extern "C"
