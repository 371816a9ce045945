// tcgen05 parameter-gradient GEMM for sm_100a, MN-major operands straight from TMA:
//   C[F_in, BD + HAB] = x^T . [d_bases | d_lin]      (dW_b = x^T d_bases, dW_c^T = x^T d_lin;
//                                                     ref: autograd of optimized_layers.py:180-182)
//
// The contraction runs over the NODE dimension and both operands are feature-contiguous in memory, i.e. MN-major.
// k_wgrad_tc (wgrad_tc.cu) transposes them through registers into the K-major no-swizzle layout - its four converter
// warps move 19 KB in and 38 KB out of shared memory per 16 nodes and bound the kernel.  Here the operands stay as they
// are: a TMA tensor copy of a [32 nodes x 32 features] box in the "128-byte span, 32-byte atom" swizzle lands exactly in
// the one MN-major layout kind::tf32 accepts, SWIZZLE_128B_BASE32B (32 contiguous features = one 128-byte row per node,
// the four 32-byte chunks of a row XOR-permuted with the row index mod 4; 4-node groups 512 B apart = SBO, 32-feature
// blocks one box apart = LBO), so the raw tile IS the hi operand (kind::tf32 ignores the low mantissa bits) and the
// converters only produce  lo = a - tf32(a)  elementwise - no transposes, half the shared-memory traffic per node.
// (The plain 16-byte-atom SWIZZLE_128B MN-major layout is rejected by the tf32 MMA: it yields zeros.)
//   warp  9     copy      one lane: 4 + ceil(n1/32) + ceil(n2/32) boxes per 32-node chunk, mbarrier transaction bytes
//   warps 5-8   convert   lo tile of the chunk (same offsets: layout-agnostic)
//   warp  4     MMA       one elected lane; per 8-node k-step: x_hi.d_hi + x_hi.d_lo + x_lo.d_hi into a 128 x N_pad fp32
//                         accumulator in TMEM (instruction descriptor: A and B MN-major)
//   warps 0-3   epilogue  every kMnSegChunks chunks the accumulator is flushed into this CTA's partial tile (fp32 adds;
//                         bounds the length of the in-TMEM accumulation); two accumulators alternate
// Accumulator columns: [0, n1) = d_bases features, [32 ceil(n1/32), ... + n2) = d_lin features (block-aligned).
// k_wgrad_reduce (wgrad_tc.cu) sums the per-CTA partial tiles deterministically.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "project.cuh"
#include "tc_common.cuh"

namespace egc {

constexpr int kMnThreads = 320;          // warps 0-3 epilogue, 4 MMA, 5-8 converters, 9 copy producer
constexpr int kMnChunk = 32;             // nodes per chunk (4 UMMA k-steps of 8)
constexpr int kMnM = 128;                // feature rows of the accumulator tile (F_in padded)
constexpr int kMnBox = 32 * kMnChunk * 4;   // one [32 nodes x 32 features] box: 4 KB
constexpr int kMnABytes = (kMnM / 32) * kMnBox;   // the A operand always spans 4 blocks
constexpr int kMnMaxSmem = 227 * 1024;
constexpr int kMnLoStages = 2;
constexpr int kMnMaxRaw = 6;
constexpr int kMnSegChunks = 12;         // chunks accumulated in TMEM between two flushes (384 nodes, as k_wgrad_tc)
constexpr int kMnConvThreads = 128;

struct MnParams {
  int f_in, n1, n2, n_nodes;
  int nb1, nb2;                          // 32-feature blocks of d_bases / d_lin
  int n_pad;                             // accumulator columns (multiple of 16): 32 * nb1 + n2 rounded up
  int n_terms;
  int raw_stages;
  int stage_bytes;                       // kMnABytes + (nb1 + nb2) * kMnBox
  int chunks_total, chunks_per_cta;
  float* partial;                        // [grid][kMnM][n_pad]
};

// MN-major tf32 operand, SWIZZLE_128B_BASE32B: 32 contiguous features per node row (128 B), swizzle atom = 4 node rows
// (512 B); SBO = distance between 4-node groups, LBO = distance between 32-feature blocks
__device__ __forceinline__ uint64_t make_desc_mn_sw128(uint32_t saddr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr >> 4) & 0x3fff);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3fff) << 16;
  d |= static_cast<uint64_t>((512u >> 4) & 0x3fff) << 32;
  d |= static_cast<uint64_t>(1) << 46;                       // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(1) << 61;                       // layout_type SWIZZLE_128B_BASE32B
  return d;
}

__global__ void __launch_bounds__(kMnThreads, 1) k_wgrad_mn(const __grid_constant__ MnParams p, const __grid_constant__ CUtensorMap tm_x,
                                                             const __grid_constant__ CUtensorMap tm_d1,
                                                             const __grid_constant__ CUtensorMap tm_d2) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5;
  const int R = p.raw_stages;
  const uint32_t stage_bytes = static_cast<uint32_t>(p.stage_bytes);
  uint8_t* raw_ring = smem;
  uint8_t* lo_ring = smem + static_cast<size_t>(R) * stage_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(lo_ring + static_cast<size_t>(kMnLoStages) * stage_bytes);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * kMnMaxRaw + kMnLoStages + 4);
  const uint32_t bar0 = smem_u32(bars);
  auto raw_full = [&](int s) { return bar0 + 8u * s; };
  auto raw_empty = [&](int s) { return bar0 + 8u * (R + s); };
  auto conv_full = [&](int s) { return bar0 + 8u * (2 * R + s); };
  auto lo_empty = [&](int s) { return bar0 + 8u * (3 * R + s); };
  auto tfull_bar = [&](int s) { return bar0 + 8u * (3 * R + kMnLoStages + s); };
  auto tempty_bar = [&](int s) { return bar0 + 8u * (3 * R + kMnLoStages + 2 + s); };

  if (tid == 0) {
    for (int s = 0; s < R; ++s) { mbar_init(raw_full(s), 1); mbar_init(raw_empty(s), 1); mbar_init(conv_full(s), kMnConvThreads); }
    for (int s = 0; s < kMnLoStages; ++s) mbar_init(lo_empty(s), 1);
    for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 128); }
    fence_barrier_init();
  }
  if (warp == 4) tmem_alloc(smem_u32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int c_begin = blockIdx.x * p.chunks_per_cta;
  const int c_end = min(c_begin + p.chunks_per_cta, p.chunks_total);
  const int n_chunks = max(c_end - c_begin, 0);
  const uint32_t raw_addr = smem_u32(raw_ring), lo_addr = smem_u32(lo_ring);
  const int n_boxes = kMnM / 32 + p.nb1 + p.nb2;

  if (warp >= 9) {
    // ================= copy producer: one box per 32 features of x / d_bases / d_lin =================
    if (warp == 9 && elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int c = c_begin; c < c_end; ++c) {
        const int node0 = c * kMnChunk;                        // rows past n_nodes are zero-filled by the TMA unit
        mbar_wait(raw_empty(stage), phase ^ 1u);
        mbar_arrive_expect_tx(raw_full(stage), static_cast<uint32_t>(n_boxes) * kMnBox);
        uint32_t dst = raw_addr + stage * stage_bytes;
        for (int b = 0; b < kMnM / 32; ++b, dst += kMnBox) tma_load_2d(dst, &tm_x, 32 * b, node0, raw_full(stage));
        for (int b = 0; b < p.nb1; ++b, dst += kMnBox) tma_load_2d(dst, &tm_d1, 32 * b, node0, raw_full(stage));
        for (int b = 0; b < p.nb2; ++b, dst += kMnBox) tma_load_2d(dst, &tm_d2, 32 * b, node0, raw_full(stage));
        if (++stage == R) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp >= 5) {
    // ================= converters: lo = a - tf32(a), same offsets as the raw tile =================
    const int ct = tid - 5 * 32;
    int stage = 0, lo = 0;
    uint32_t phase = 0, lo_phase = 0;
    for (int c = 0; c < n_chunks; ++c) {
      mbar_wait(raw_full(stage), phase);
      mbar_wait(lo_empty(lo), lo_phase ^ 1u);
      const uint32_t src = raw_addr + stage * stage_bytes, dst = lo_addr + lo * stage_bytes;
      if (p.n_terms == 3) {
        for (uint32_t off = ct * 16; off < stage_bytes; off += kMnConvThreads * 16 * 4) {
          float4 v[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const uint32_t o = off + u * (kMnConvThreads * 16);
            v[u] = o < stage_bytes ? lds128(src + o) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const uint32_t o = off + u * (kMnConvThreads * 16);
            if (o < stage_bytes)
              sts128(dst + o, make_float4(v[u].x - tf32_hi(v[u].x), v[u].y - tf32_hi(v[u].y), v[u].z - tf32_hi(v[u].z),
                                          v[u].w - tf32_hi(v[u].w)));
          }
        }
        fence_proxy_async();
      }
      mbar_arrive(conv_full(stage));
      if (++stage == R) { stage = 0; phase ^= 1u; }
      if (++lo == kMnLoStages) { lo = 0; lo_phase ^= 1u; }
    }
  } else if (warp == 4) {
    // ================= MMA issuer: converged warp, uniform descriptors, one elected lane issues =================
    const uint32_t tmem_u = __shfl_sync(kFull, tmem_base, 0);
    // c f32, a / b tf32, A and B MN-major (bits 15 / 16), N >> 3, M >> 4
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) |
                           (static_cast<uint32_t>(p.n_pad >> 3) << 17) | (static_cast<uint32_t>(kMnM >> 4) << 24);
    const uint64_t da_raw0 = make_desc_mn_sw128(raw_addr, kMnBox), db_raw0 = make_desc_mn_sw128(raw_addr + kMnABytes, kMnBox);
    const uint64_t da_lo0 = make_desc_mn_sw128(lo_addr, kMnBox), db_lo0 = make_desc_mn_sw128(lo_addr + kMnABytes, kMnBox);
    const bool three = p.n_terms == 3;
    const bool leader = elect_one();
    int stage = 0, lo = 0;
    uint32_t phase = 0;
    int seg = 0;
    for (int c = 0; c < n_chunks; ++seg) {
      const int acc = seg & 1;
      mbar_wait(tempty_bar(acc), ((static_cast<uint32_t>(seg) >> 1) & 1u) ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_u + static_cast<uint32_t>(acc) * 256u;
      const int seg_end = min(c + kMnSegChunks, n_chunks);
      for (int first = 1; c < seg_end; ++c, first = 0) {
        mbar_wait(conv_full(stage), phase);
        tc_fence_after();
        if (leader) {
          const uint32_t so = static_cast<uint32_t>(stage) * (stage_bytes >> 4), lo_o = static_cast<uint32_t>(lo) * (stage_bytes >> 4);
#pragma unroll
          for (int s = 0; s < kMnChunk / 8; ++s) {               // 8 nodes per k-step: the next 1 KB group
            const uint32_t ko = s * (1024u >> 4);
            umma_tf32(d_tmem, da_raw0 + (so + ko), db_raw0 + (so + ko), idesc, (first && s == 0) ? 0u : 1u);
            if (three) {
              umma_tf32(d_tmem, da_raw0 + (so + ko), db_lo0 + (lo_o + ko), idesc, 1u);
              umma_tf32(d_tmem, da_lo0 + (lo_o + ko), db_raw0 + (so + ko), idesc, 1u);
            }
          }
          umma_commit(raw_empty(stage));
          umma_commit(lo_empty(lo));
          if (c + 1 == seg_end) umma_commit(tfull_bar(acc));
        }
        __syncwarp();
        if (++stage == R) { stage = 0; phase ^= 1u; }
        if (++lo == kMnLoStages) lo = 0;
      }
    }
  } else {
    // ================= epilogue: flush each segment into this CTA's partial tile =================
    float* dst = p.partial + (static_cast<int64_t>(blockIdx.x) * kMnM + tid) * p.n_pad;
    if (n_chunks == 0) {
      for (int col = 0; col < p.n_pad; col += 4) *reinterpret_cast<float4*>(dst + col) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const uint32_t lane_base = static_cast<uint32_t>(warp * 32) << 16;
    int seg = 0;
    for (int c = 0; c < n_chunks; c += kMnSegChunks, ++seg) {
      const int acc = seg & 1;
      mbar_wait(tfull_bar(acc), (static_cast<uint32_t>(seg) >> 1) & 1u);
      tc_fence_after();
      for (int col0 = 0; col0 < p.n_pad; col0 += 16) {
        uint32_t r[16];
        tmem_ld16(tmem_base + lane_base + static_cast<uint32_t>(acc) * 256u + static_cast<uint32_t>(col0), r);
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float4 v = make_float4(__uint_as_float(r[4 * q]), __uint_as_float(r[4 * q + 1]), __uint_as_float(r[4 * q + 2]),
                                 __uint_as_float(r[4 * q + 3]));
          float4* d4 = reinterpret_cast<float4*>(dst + col0 + 4 * q);
          if (seg > 0) { const float4 o = *d4; v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w; }
          *d4 = v;
        }
      }
      tc_fence_before();
      mbar_arrive(tempty_bar(acc));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, 512);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
typedef CUresult (*MnEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static MnEncodeTiledFn mn_encode_tiled() {
  static MnEncodeTiledFn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
      f = nullptr;
    return reinterpret_cast<MnEncodeTiledFn>(f);
  }();
  return fn;
}

// [n_nodes rows x width floats] with a row pitch of ld floats, boxes of 32 nodes x 32 features, 128-byte span / 32-byte atom
// swizzle; columns past `width` read as zeros (a column range of a wider matrix: base = first column, ld = full width)
static bool make_mn_map(CUtensorMap* m, const float* base, int width, int ld, int n_nodes) {
  MnEncodeTiledFn fn = mn_encode_tiled();
  if (fn == nullptr || base == nullptr || width <= 0) return false;
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(width), static_cast<cuuint64_t>(n_nodes)};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 4};
  const cuuint32_t box[2] = {32, static_cast<cuuint32_t>(kMnChunk)};
  const cuuint32_t es[2] = {1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static int mn_round16(int v) { return (v + 15) / 16 * 16; }
static int mn_n_pad(int bd, int hab) { return mn_round16(32 * ceil_div(bd, 32) + hab); }
static int mn_stage_bytes(int bd, int hab) { return kMnABytes + (ceil_div(bd, 32) + ceil_div(hab, 32)) * kMnBox; }
static int mn_raw_stages(int bd, int hab) {
  const size_t stage = static_cast<size_t>(mn_stage_bytes(bd, hab));
  const size_t fixed = kMnLoStages * stage + (3 * kMnMaxRaw + kMnLoStages + 4) * 8 + 64 + 1024;
  if (fixed + 2 * stage > static_cast<size_t>(kMnMaxSmem)) return 0;
  return static_cast<int>(std::min<size_t>(kMnMaxRaw, (kMnMaxSmem - fixed) / stage));
}

// Wide layers (more than 256 accumulator columns, e.g. REGConv's paper type: d_lin carries the combination weights of the
// root term and of every relation): the columns are cut into launches of <= 256 - the first takes d_bases and the leading
// d_lin columns, the others 256 d_lin columns each (x is streamed once per launch).
static int mn_first_lin_cols(int bd, int hab) {
  if (mn_n_pad(bd, hab) <= 256) return hab;
  return std::max(0, (256 - 32 * ceil_div(bd, 32)) / 32 * 32);
}

bool wgrad_mn_supported(int n, int f_in, int bd, int hab) {
  static const bool off = getenv("EGC_WGRAD_TRANSPOSE") != nullptr;       // A/B: keep the transposing kernel
  if (off || n < 1 || f_in % 4 || bd % 4 || hab % 4 || f_in > kMnM || hab < 1 || mn_encode_tiled() == nullptr) return false;
  const int first = mn_first_lin_cols(bd, hab);
  if (first < hab && (first < 32 || mn_raw_stages(0, std::min(hab - first, 256)) < 2)) return false;
  return mn_raw_stages(bd, first) >= 2;
}

size_t wgrad_mn_workspace(int n, int f_in, int bd, int hab) {
  (void)n; (void)f_in;
  return static_cast<size_t>(sm_count()) * kMnM * std::min(256, mn_n_pad(bd, hab)) * sizeof(float) + 256;
}

// one launch: C[F_in, n1 + n2] = x^T . [d1 | d2], d1 / d2 column ranges with row pitches ld1 / ld2 (n1 may be 0)
static int wgrad_mn_part(const float* x, const float* d1, int n1, int ld1, const float* d2, int n2, int ld2, int n, int f_in,
                         float* d_w_bases, float* d_w_comb, int n_terms, void* workspace, cudaStream_t st) {
  MnParams p{};
  p.f_in = f_in; p.n1 = n1; p.n2 = n2; p.n_nodes = n;
  p.nb1 = ceil_div(n1, 32); p.nb2 = ceil_div(n2, 32);
  p.n_pad = mn_n_pad(n1, n2);
  p.n_terms = n_terms;
  p.raw_stages = mn_raw_stages(n1, n2);
  EGC_REQUIRE(p.n_pad <= 256 && p.raw_stages >= 2, "wgrad_mn: shape does not fit the accumulator / shared memory");
  p.stage_bytes = mn_stage_bytes(n1, n2);
  p.chunks_total = ceil_div(n, kMnChunk);
  const int grid = std::min(sm_count(), p.chunks_total);
  p.chunks_per_cta = ceil_div(p.chunks_total, grid);
  p.partial = static_cast<float*>(workspace);
  alignas(64) CUtensorMap tmx, tm1, tm2;
  memset(&tmx, 0, sizeof(tmx)); memset(&tm1, 0, sizeof(tm1)); memset(&tm2, 0, sizeof(tm2));
  EGC_REQUIRE(make_mn_map(&tmx, x, f_in, f_in, n) && make_mn_map(&tm2, d2, n2, ld2, n) &&
              (n1 == 0 || make_mn_map(&tm1, d1, n1, ld1, n)), "wgrad_mn: tensor-map encoding failed");
  if (n1 == 0) tm1 = tm2;                                      // never used: no d1 boxes are issued
  const size_t smem = static_cast<size_t>(p.raw_stages + kMnLoStages) * p.stage_bytes + (3 * kMnMaxRaw + kMnLoStages + 4) * 8 + 64 + 1024;
  static bool attr_set[kMaxDevices] = {};
  EGC_CUDA(max_dynamic_smem_once(reinterpret_cast<const void*>(k_wgrad_mn), kMnMaxSmem, attr_set));
  {
    LaunchScope ls("k_wgrad_tc", st);
    k_wgrad_mn<<<grid, kMnThreads, smem, st>>>(p, tmx, tm1, tm2);
  }
  EGC_LAUNCH_CHECK("k_wgrad_mn");
  return wgrad_reduce(p.partial, grid, f_in, n1, n2, p.n_pad, 32 * p.nb1, d_w_bases, d_w_comb, st);
}

int wgrad_mn(const float* x, const float* d_bases, const float* d_lin, int n, int f_in, int bd, int hab,
             float* d_w_bases, float* d_w_comb, int n_terms, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  EGC_REQUIRE(workspace_bytes >= wgrad_mn_workspace(n, f_in, bd, hab), "wgrad_mn: workspace too small");
  const int first = mn_first_lin_cols(bd, hab);
  if (int rc = wgrad_mn_part(x, d_bases, bd, bd, d_lin, first, hab, n, f_in, d_w_bases, d_w_comb, n_terms, workspace, st)) return rc;
  for (int c0 = first; c0 < hab; c0 += 256) {                  // stream-ordered: the partial tiles are reused
    const int cols = std::min(256, hab - c0);
    if (int rc = wgrad_mn_part(x, nullptr, 0, 0, d_lin + c0, cols, hab, n, f_in, nullptr,
                               d_w_comb != nullptr ? d_w_comb + static_cast<int64_t>(c0) * f_in : nullptr, n_terms, workspace, st))
      return rc;
  }
  return EGC_OK;
}

}  // namespace egc
