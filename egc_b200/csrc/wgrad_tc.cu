// tcgen05 parameter-gradient GEMM for sm_100a:  C[F_in, BD + HAB] = x^T . [d_bases | d_lin]
// (dW_b = x^T d_bases, dW_c^T = x^T d_lin; ref: autograd of optimized_layers.py:180-182).
//
// The contraction runs over the NODE dimension, so both operands stream and both are feature-contiguous
// in memory (MN-major).  kind::tf32 MMAs only accept MN-major operands in the 128B/32B-atom swizzle
// (tools/umma_probe.cu: the no-swizzle MN-major bits yield zeros), so the operands are transposed on the
// way through shared memory instead, and the MMA sees the plain K-major no-swizzle layout:
//   warp  9     copy      one lane issues three TMA bulk copies per 16-node chunk (the x, d_bases and d_lin rows of
//                         16 consecutive nodes are each one contiguous span) into a deep ring of
//                         [x | d_bases | d_lin] blocks; completion lands on an mbarrier as transaction bytes
//   warps 5-8   convert   4 nodes x 4 features register transposes -> hi / lo split -> the canonical K-major
//                         layout (8 rows x 16 B core matrices, K = node), conflict-free rotated stores
//   warp  4     MMA       one elected lane, 3-term split into a 128 x N_pad fp32 accumulator in TMEM
//   warps 0-3   epilogue  every kSegChunks chunks the accumulator is flushed into this CTA's partial tile
//                         in global memory (fp32 RN adds; bounds the length of the in-TMEM accumulation);
//                         two accumulators alternate so the flush overlaps the next segment's MMAs
// Each persistent CTA owns a contiguous range of 16-node chunks; a small deterministic kernel reduces the
// per-CTA partial tiles into dW_b / dW_c (transposing the latter).
#include <algorithm>

#include "project.cuh"
#include "tc_common.cuh"

namespace egc {

constexpr int kWgThreads = 320;          // warps 0-3 epilogue, 4 MMA, 5-8 converters, 9 copy producer
constexpr int kWgChunk = 16;             // nodes per chunk (2 UMMA k-steps)
constexpr int kWgM = 128;                // feature rows of the accumulator tile (F_in padded)
constexpr int kWgMaxSmem = 227 * 1024;
constexpr int kWgOpStages = 2;
constexpr int kWgMaxRaw = 12;
constexpr int kSegChunks = 24;           // chunks accumulated in TMEM between two flushes (384 nodes)
constexpr int kWgConvThreads = 128;

struct WgParams {
  const float* x; int f_in;              // A^T source: x[n, f_in]
  const float* d1; int n1;               // B source, columns [0, n1)      : d_bases[n, n1]
  const float* d2; int n2;               // B source, columns [n1, n1+n2)  : d_lin[n, n2]
  int n_nodes;
  int n_pad;                             // multiple of 16
  int n_terms;
  int raw_stages;
  int chunks_total, chunks_per_cta;
  uint32_t ppn_magic;                    // ceil(2^32 / pieces_per_node)
  float* partial;                        // [grid][kWgM][n_pad]
};

__global__ void __launch_bounds__(kWgThreads, 1) k_wgrad_tc(const __grid_constant__ WgParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5;
  const int W = p.f_in + p.n1 + p.n2;                                // floats per raw node row
  const int ppn = W >> 2;                                            // 16-byte pieces per node
  const uint32_t a_half = kWgM * kWgChunk * 4;                       // 8 KB: hi (or lo) of an A chunk
  const uint32_t b_half = static_cast<uint32_t>(p.n_pad) * kWgChunk * 4;
  const uint32_t op_bytes = 2 * (a_half + b_half);                   // [A_hi | A_lo | B_hi | B_lo]
  const uint32_t raw_bytes = static_cast<uint32_t>(kWgChunk) * W * 4;
  const int R = p.raw_stages;
  uint8_t* op_ring = smem;
  uint8_t* raw_ring = smem + kWgOpStages * op_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(raw_ring + static_cast<size_t>(R) * raw_bytes);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kWgMaxRaw + 8);
  const uint32_t bar0 = smem_u32(bars);
  auto raw_full = [&](int s) { return bar0 + 8u * s; };
  auto raw_empty = [&](int s) { return bar0 + 8u * (R + s); };
  auto op_full = [&](int s) { return bar0 + 8u * (2 * R + s); };
  auto op_empty = [&](int s) { return bar0 + 8u * (2 * R + 2 + s); };
  auto tfull_bar = [&](int s) { return bar0 + 8u * (2 * R + 4 + s); };
  auto tempty_bar = [&](int s) { return bar0 + 8u * (2 * R + 6 + s); };

  if (tid == 0) {
    for (int s = 0; s < R; ++s) { mbar_init(raw_full(s), 1); mbar_init(raw_empty(s), kWgConvThreads); }
    for (int s = 0; s < 2; ++s) {
      mbar_init(op_full(s), kWgConvThreads); mbar_init(op_empty(s), 1);
      mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 128);
    }
    fence_barrier_init();
  }
  if (warp == 4) tmem_alloc(smem_u32(tmem_slot), 512);
  // operand rows beyond f_in / n1 + n2 are never written by the converters: zero them once
  for (uint32_t off = tid * 16; off < kWgOpStages * op_bytes; off += kWgThreads * 16)
    *reinterpret_cast<float4*>(op_ring + off) = make_float4(0.f, 0.f, 0.f, 0.f);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int c_begin = blockIdx.x * p.chunks_per_cta;
  const int c_end = min(c_begin + p.chunks_per_cta, p.chunks_total);
  const int n_chunks = max(c_end - c_begin, 0);
  const uint32_t a_lbo = kWgM * 16, b_lbo = static_cast<uint32_t>(p.n_pad) * 16;   // bytes between 4-node K pieces
  const uint32_t raw_addr = smem_u32(raw_ring), op_addr = smem_u32(op_ring);

  if (warp >= 9) {
    // ================= copy producer: three bulk copies per chunk =================
    const bool leader = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    for (int c = c_begin; c < c_end; ++c) {
      const int64_t node0 = static_cast<int64_t>(c) * kWgChunk;
      const uint32_t valid = static_cast<uint32_t>(min(static_cast<int64_t>(kWgChunk), p.n_nodes - node0));
      const uint32_t bx = valid * p.f_in * 4, b1 = valid * p.n1 * 4, b2 = valid * p.n2 * 4;
      mbar_wait(raw_empty(stage), phase ^ 1u);
      if (leader) {
        const uint32_t dst = raw_addr + stage * raw_bytes;
        mbar_arrive_expect_tx(raw_full(stage), bx + b1 + b2);
        bulk_g2s(dst, p.x + node0 * p.f_in, bx, raw_full(stage));
        bulk_g2s(dst + kWgChunk * p.f_in * 4, p.d1 + node0 * p.n1, b1, raw_full(stage));
        if (b2 > 0) bulk_g2s(dst + kWgChunk * (p.f_in + p.n1) * 4, p.d2 + node0 * p.n2, b2, raw_full(stage));
      }
      __syncwarp();
      if (++stage == R) { stage = 0; phase ^= 1u; }
    }
  } else if (warp >= 5) {
    // ================= converters: transpose 4 nodes x 4 features, hi / lo split =================
    const int ct = tid - 5 * 32;
    const int n_blocks = 4 * ppn;                          // (node quad, feature quad) blocks per chunk
    const uint32_t off_d1 = kWgChunk * p.f_in * 4, off_d2 = kWgChunk * (p.f_in + p.n1) * 4;
    int stage = 0, op = 0;
    uint32_t phase = 0, op_phase = 0;
    for (int c = 0; c < n_chunks; ++c) {
      mbar_wait(raw_full(stage), phase);
      mbar_wait(op_empty(op), op_phase ^ 1u);
      const uint32_t src0 = raw_addr + stage * raw_bytes;
      const uint32_t dst0 = op_addr + op * op_bytes;
      // nodes of this chunk that exist (the bulk copies of the last chunk stop at the end of the arrays)
      const int valid = min(kWgChunk, p.n_nodes - (c_begin + c) * kWgChunk);
      for (int b = ct; b < n_blocks; b += kWgConvThreads) {
        const int quad = static_cast<int>(__umulhi(static_cast<uint32_t>(b), p.ppn_magic));    // b / ppn
        const int fq = b - quad * ppn;
        const int f = fq * 4;
        uint32_t src, row_bytes;                           // block of 4 nodes x 4 features inside its region
        if (f < p.f_in) { row_bytes = p.f_in * 4; src = src0 + f * 4; }
        else if (f < p.f_in + p.n1) { row_bytes = p.n1 * 4; src = src0 + off_d1 + (f - p.f_in) * 4; }
        else { row_bytes = p.n2 * 4; src = src0 + off_d2 + (f - p.f_in - p.n1) * 4; }
        src += static_cast<uint32_t>(quad) * 4 * row_bytes;
        float4 v0 = lds128(src), v1 = lds128(src + row_bytes), v2 = lds128(src + 2 * row_bytes),
               v3 = lds128(src + 3 * row_bytes);
        if (valid < kWgChunk) {
          const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
          const int n0 = quad * 4;
          if (n0 >= valid) v0 = z;
          if (n0 + 1 >= valid) v1 = z;
          if (n0 + 2 >= valid) v2 = z;
          if (n0 + 3 >= valid) v3 = z;
        }
        float4 o[4] = {make_float4(v0.x, v1.x, v2.x, v3.x), make_float4(v0.y, v1.y, v2.y, v3.y),
                       make_float4(v0.z, v1.z, v2.z, v3.z), make_float4(v0.w, v1.w, v2.w, v3.w)};
        // rotate the store order by (fq / 2) % 4 so that the 8 lanes of a store phase hit 8 distinct 16-byte bank groups
        const int rot = (fq >> 1) & 3;
        if (rot & 1) { const float4 t = o[0]; o[0] = o[1]; o[1] = o[2]; o[2] = o[3]; o[3] = t; }
        if (rot & 2) { float4 t = o[0]; o[0] = o[2]; o[2] = t; t = o[1]; o[1] = o[3]; o[3] = t; }
        uint32_t dst, lo_off;
        if (f < p.f_in) { dst = dst0 + quad * a_lbo + f * 16; lo_off = a_half; }
        else { dst = dst0 + 2 * a_half + quad * b_lbo + (f - p.f_in) * 16; lo_off = b_half; }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint32_t d = dst + ((i + rot) & 3) * 16;
          const float4 h = make_float4(tf32_hi(o[i].x), tf32_hi(o[i].y), tf32_hi(o[i].z), tf32_hi(o[i].w));
          const float4 l = make_float4(o[i].x - h.x, o[i].y - h.y, o[i].z - h.z, o[i].w - h.w);
          sts128(d, h);
          sts128(d + lo_off, l);
        }
      }
      mbar_arrive(raw_empty(stage));
      fence_proxy_async();
      mbar_arrive(op_full(op));
      if (++stage == R) { stage = 0; phase ^= 1u; }
      if (++op == kWgOpStages) { op = 0; op_phase ^= 1u; }
    }
  } else if (warp == 4) {
    // ================= MMA issuer: converged warp, uniform descriptors, one elected lane issues =================
    const uint32_t tmem_u = __shfl_sync(kFull, tmem_base, 0);
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(p.n_pad >> 3) << 17) |
                           (static_cast<uint32_t>(kWgM >> 4) << 24);
    const uint64_t da0 = make_desc(op_addr, a_lbo, 128), db0 = make_desc(op_addr + 2 * a_half, b_lbo, 128);
    const uint32_t a_lo_off = a_half >> 4, b_lo_off = b_half >> 4;
    const uint32_t a_kstep = (2 * a_lbo) >> 4, b_kstep = (2 * b_lbo) >> 4;
    const bool three = p.n_terms == 3;
    const bool leader = elect_one();
    int op = 0;
    uint32_t op_phase = 0;
    int seg = 0;
    for (int c = 0; c < n_chunks; ++seg) {
      const int acc = seg & 1;
      mbar_wait(tempty_bar(acc), ((static_cast<uint32_t>(seg) >> 1) & 1u) ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_u + static_cast<uint32_t>(acc) * 256u;
      const int seg_end = min(c + kSegChunks, n_chunks);
      for (int first = 1; c < seg_end; ++c, first = 0) {
        mbar_wait(op_full(op), op_phase);
        tc_fence_after();
        if (leader) {
          const uint32_t so = static_cast<uint32_t>(op) * (op_bytes >> 4);
#pragma unroll
          for (int s = 0; s < 2; ++s) {
            const uint64_t da_hi = da0 + (so + s * a_kstep), db_hi = db0 + (so + s * b_kstep);
            umma_tf32(d_tmem, da_hi, db_hi, idesc, (first && s == 0) ? 0u : 1u);
            if (three) {
              umma_tf32(d_tmem, da_hi, db_hi + b_lo_off, idesc, 1u);
              umma_tf32(d_tmem, da_hi + a_lo_off, db_hi, idesc, 1u);
            }
          }
          umma_commit(op_empty(op));
          if (c + 1 == seg_end) umma_commit(tfull_bar(acc));
        }
        __syncwarp();
        if (++op == kWgOpStages) { op = 0; op_phase ^= 1u; }
      }
    }
  } else {
    // ================= epilogue: flush each segment into this CTA's partial tile =================
    float* dst = p.partial + (static_cast<int64_t>(blockIdx.x) * kWgM + tid) * p.n_pad;
    if (n_chunks == 0) {
      for (int col = 0; col < p.n_pad; col += 4) *reinterpret_cast<float4*>(dst + col) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const uint32_t lane_base = static_cast<uint32_t>(warp * 32) << 16;
    int seg = 0;
    for (int c = 0; c < n_chunks; c += kSegChunks, ++seg) {
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

// dW_b[m][n] = sum_cta partial[cta][m][n] (n < n1);  dW_c[n - n1][m] = sum_cta partial[cta][m][n] (n >= n1)
// A block owns 32 consecutive outputs; its 8 warps sum interleaved subsets of the per-CTA partials (4 independent
// accumulators each) and warp 0 adds the 8 sub-sums in a fixed order: deterministic, and ~5 dependent load rounds
// instead of the 37 of a one-thread-per-output walk over 148 partials (23 us -> a few us).
constexpr int kWgRedSplit = 8;
__global__ void __launch_bounds__(32 * kWgRedSplit) k_wgrad_reduce(const float* __restrict__ partial, int n_cta, int f_in, int n1,
                                                                    int n2, int n_pad, int n2_col0, float* __restrict__ d_w_bases,
                                                                    float* __restrict__ d_w_comb) {
  __shared__ float sub[kWgRedSplit][32];
  const int lane = threadIdx.x & 31, s = threadIdx.x >> 5;
  const int idx = blockIdx.x * 32 + lane;
  const int N = n1 + n2;
  const bool ok = idx < f_in * N;
  const int m = ok ? idx / N : 0, n = ok ? idx - m * N : 0;
  const float* src = partial + static_cast<int64_t>(m) * n_pad + (n < n1 ? n : n2_col0 + (n - n1));
  const int64_t stride = static_cast<int64_t>(kWgM) * n_pad;
  float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
  if (ok) {
    int c = s;
    for (; c + 3 * kWgRedSplit < n_cta; c += 4 * kWgRedSplit) {
      t0 += src[c * stride]; t1 += src[(c + kWgRedSplit) * stride];
      t2 += src[(c + 2 * kWgRedSplit) * stride]; t3 += src[(c + 3 * kWgRedSplit) * stride];
    }
    for (; c < n_cta; c += kWgRedSplit) t0 += src[c * stride];
  }
  sub[s][lane] = (t0 + t1) + (t2 + t3);
  __syncthreads();
  if (s != 0 || !ok) return;
  float t = 0.f;
#pragma unroll
  for (int k = 0; k < kWgRedSplit; ++k) t += sub[k][lane];
  if (n < n1) { if (d_w_bases != nullptr) d_w_bases[static_cast<int64_t>(m) * n1 + n] = t; }
  else if (d_w_comb != nullptr) d_w_comb[static_cast<int64_t>(n - n1) * f_in + m] = t;
}

int wgrad_reduce(const float* partial, int n_cta, int f_in, int n1, int n2, int n_pad, int n2_col0, float* d_w_bases,
                 float* d_w_comb, cudaStream_t st) {
  const int total = f_in * (n1 + n2);
  {
    LaunchScope ls("k_wgrad_reduce", st);
    k_wgrad_reduce<<<ceil_div(total, 32), 32 * kWgRedSplit, 0, st>>>(partial, n_cta, f_in, n1, n2, n_pad, n2_col0, d_w_bases, d_w_comb);
  }
  EGC_LAUNCH_CHECK("k_wgrad_reduce");
  return EGC_OK;
}

static int round16w(int v) { return (v + 15) / 16 * 16; }

static int wgrad_raw_stages(int f_in, int n_pad, int width) {
  const size_t op = 2 * (static_cast<size_t>(kWgM) * kWgChunk * 4 + static_cast<size_t>(n_pad) * kWgChunk * 4);
  const size_t raw = static_cast<size_t>(kWgChunk) * width * 4;
  const size_t fixed = kWgOpStages * op + (2 * kWgMaxRaw + 8) * 8 + 64;
  (void)f_in;
  if (fixed + 2 * raw > static_cast<size_t>(kWgMaxSmem)) return 0;
  return static_cast<int>(std::min<size_t>(kWgMaxRaw, (kWgMaxSmem - fixed) / raw));
}

bool wgrad_tc_supported(int n, int f_in, int bd, int hab) {
  if (n < 1 || f_in % 4 || bd % 4 || hab % 4 || f_in > kWgM) return false;
  const int n_pad = round16w(bd + hab);
  return n_pad <= 256 && wgrad_raw_stages(f_in, n_pad, f_in + bd + hab) >= 2;
}

size_t wgrad_tc_workspace(int n, int f_in, int bd, int hab) {
  (void)n; (void)f_in;
  return static_cast<size_t>(sm_count()) * kWgM * round16w(bd + hab) * sizeof(float) + 256;
}

int wgrad_tc(const float* x, const float* d_bases, const float* d_lin, int n, int f_in, int bd, int hab,
             float* d_w_bases, float* d_w_comb, int n_terms, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  EGC_REQUIRE(workspace_bytes >= wgrad_tc_workspace(n, f_in, bd, hab), "wgrad_tc: workspace too small");
  WgParams p{};
  p.x = x; p.f_in = f_in; p.d1 = d_bases; p.n1 = bd; p.d2 = d_lin; p.n2 = hab; p.n_nodes = n;
  p.n_pad = round16w(bd + hab);
  p.n_terms = n_terms;
  const int width = f_in + bd + hab;
  p.raw_stages = wgrad_raw_stages(f_in, p.n_pad, width);
  EGC_REQUIRE(p.raw_stages >= 2, "wgrad_tc: shape does not fit shared memory");
  p.chunks_total = ceil_div(n, kWgChunk);
  const int grid = std::min(sm_count(), p.chunks_total);
  p.chunks_per_cta = ceil_div(p.chunks_total, grid);
  const uint32_t ppn = static_cast<uint32_t>(width / 4);
  p.ppn_magic = static_cast<uint32_t>((0x100000000ull + ppn - 1) / ppn);
  p.partial = static_cast<float*>(workspace);
  const size_t op = 2 * (static_cast<size_t>(kWgM) * kWgChunk * 4 + static_cast<size_t>(p.n_pad) * kWgChunk * 4);
  const size_t smem = kWgOpStages * op + static_cast<size_t>(p.raw_stages) * kWgChunk * width * 4 + (2 * kWgMaxRaw + 8) * 8 + 64;
  static bool attr_set[kMaxDevices] = {};
  EGC_CUDA(max_dynamic_smem_once(reinterpret_cast<const void*>(k_wgrad_tc), kWgMaxSmem, attr_set));
  {
    LaunchScope ls("k_wgrad_tc", st);
    k_wgrad_tc<<<grid, kWgThreads, smem, st>>>(p);
  }
  EGC_LAUNCH_CHECK("k_wgrad_tc");
  return wgrad_reduce(p.partial, grid, f_in, bd, hab, p.n_pad, bd, d_w_bases, d_w_comb, st);
}

}  // namespace egc
