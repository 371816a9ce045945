// tcgen05 (5th-gen tensor core) projections for sm_100a:  C[M, N] = [A1 | A2][M, K] . B[K, N]
//
//   forward : [bases | weightings] = x . [W_b | W_c^T]   (+ bias, sigmoid on the weightings columns)
//   backward: d_x = [d_bases | d_lin] . [W_b | W_c^T]^T
//
// fp32 parity through kind::tf32 MMAs comes from the 3-term split  a.b ~= ah.bh + ah.bl + al.bh  with
// ah = a & 0xffffe000 (exact TF32), al = a - ah, accumulated in fp32 in TMEM (n_terms = 1 gives plain TF32).
//
// The op is an HBM stream (AI ~ 37 flop/B), so the kernel is organised around bytes in flight:
// one persistent CTA per SM, 11 warps:
//   warps 9-10  copy      default: one lane of warp 9 issues TMA tensor copies - four [128 rows x 16 B] boxes per 8 KB
//                         chunk, each landing as 16 stacked core matrices, completion by mbarrier transaction bytes.
//                         Fallback (no tensor-map encoder / unaligned rows):
//                         cp.async (16 B, L2-only) of raw A chunks into a deep shared-memory ring, already in
//                         the canonical K-major no-swizzle UMMA layout (8-row x 16-byte core matrices);
//                         completion is signalled on an mbarrier (cp.async.mbarrier.arrive.noinc), so up to
//                         `raw_stages` x 8 KB per SM are in flight without holding registers
//   warps 5-8   convert   raw chunk -> hi (in place) and lo (2-deep side ring), fence.proxy.async
//   warp  4     MMA       one elected lane issues tcgen05.mma / tcgen05.commit; owns the TMEM allocation
//   warps 0-3   epilogue  tcgen05.ld of the 128 x N accumulator (TMEM lanes 32w..32w+31) -> global
// The weights (B, hi and lo) are staged once per CTA and stay resident in shared memory.  When B (hi + lo)
// would leave too little room for the A ring, the output columns are split over `n_split` groups of CTAs
// (CTA c serves group c % n_split); the groups walk the row tiles in lockstep, so the second read of an A
// tile is an L2 hit.  The accumulator is double-buffered in TMEM (2 x 256 columns): the epilogue of tile t
// overlaps the main loop of tile t+1.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "bf16.cuh"
#include "project.cuh"
#include "tc_common.cuh"

namespace egc {

constexpr int kTcThreads = 352;
constexpr int kTileM = 128;
constexpr int kChunkK = 16;                                   // floats of K per A chunk (2 UMMA k-steps of 8)
constexpr int kChunkBytes = kTileM * kChunkK * 4;             // 8 KB (raw / hi, or lo)
constexpr int kLoStages = 4;
constexpr int kMaxRawStages = 16;
constexpr int kCopyWarps = 2;
constexpr int kConvWarps = 4;                                 // == kLoStages: converter warp w owns lo slot w
constexpr int kEpiRowBytes = 144;                             // 32 floats + 16 B pad: conflict-free row-per-thread stores
constexpr int kEpiStageBytes = 4 * 32 * kEpiRowBytes;         // one 32 x 32 staging tile per epilogue warp
constexpr int kMaxSmem = 227 * 1024;
constexpr int kTmemCols = 512;

struct TcParams {
  const float* a1; int lda1; int k1;      // A = [a1 | a2], row-major
  const float* a2; int lda2; int k2;
  int M;
  // B(n, k) = b[nb][kb][ (n - n_off) * sn + (k - k_off) * sk ],  nb = n >= n1, kb = k >= k1
  const float* b[2][2];
  int b_sn[2][2], b_sk[2][2];
  int n1, n2;                              // N = n1 + n2; columns >= n1 go to c2
  float* c1; int ldc1;
  float* c2; int ldc2;
  const float* bias2;
  int sigmoid2;
  int k_pad;                               // multiple of 16
  int n_split, cols_per_group;             // output columns [g * cols_per_group, ...) belong to CTA group g
  int raw_stages;
  int n_terms;                             // 3: 3xTF32, 1: TF32
  int num_tiles;
  int use_tma_store;                       // epilogue writes C through TMA tensor stores (128B-swizzled 32 x 32 staging tiles)
  int use_tma;                             // A chunks arrive by TMA tensor copies instead of LDGSTS: 1 = four [128 rows x 16 B]
                                           // boxes per chunk (no-swizzle core matrices), 2 = ONE [128 rows x 64 B] box per
                                           // chunk in the 64-byte swizzle (4x fewer, 4x wider requests)
  int ablate;                              // diagnostics (EGC_TC_ABLATE, results become wrong): 1 no lo conversion, 2 no epilogue,
                                           // 4 no MMA, 8 no A copies, 16 no global stores  (tools/gemm_ablate.sh)
};

// ---------------------------------------------------------------------------------------------
// kernel
// ---------------------------------------------------------------------------------------------
// BF16_C1: the columns of c1 (the basis rows of the forward) are rounded to bf16 (nearest even) in the epilogue and stored
// packed - c1 then points at bf16 rows; c2 (the weightings) stays fp32.  The TMA-store epilogue is not used with it.
template <bool BF16_C1>
__global__ void __launch_bounds__(kTcThreads, 1) k_project_tc(const __grid_constant__ TcParams p, const __grid_constant__ CUtensorMap tm_a1,
                                                               const __grid_constant__ CUtensorMap tm_a2, const __grid_constant__ CUtensorMap tm_c1,
                                                               const __grid_constant__ CUtensorMap tm_c2) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int K = p.k1 + p.k2, N = p.n1 + p.n2;
  const int R = p.raw_stages;
  const int group = blockIdx.x % p.n_split;
  const int n_begin = group * p.cols_per_group;
  const int n_count = min(p.cols_per_group, N - n_begin);
  const int n_pad = (n_count + 15) & ~15;
  const uint32_t b_half_bytes = static_cast<uint32_t>(p.cols_per_group) * p.k_pad * 4;
  const uint32_t lbo_b = static_cast<uint32_t>(n_pad) * 16;              // bytes between 16-byte K pieces of B
  uint8_t* b_hi = smem;
  uint8_t* b_lo = smem + b_half_bytes;
  uint8_t* lo_ring = smem + 2 * b_half_bytes;
  uint8_t* epi_stage = lo_ring + kLoStages * kChunkBytes;
  uint8_t* raw_ring = epi_stage + kEpiStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(raw_ring + static_cast<size_t>(R) * kChunkBytes);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * kMaxRawStages + kLoStages + 4);
  const uint32_t bar0 = smem_u32(bars);
  auto raw_full = [&](int s) { return bar0 + 8u * s; };
  auto raw_empty = [&](int s) { return bar0 + 8u * (R + s); };
  auto conv_full = [&](int s) { return bar0 + 8u * (2 * R + s); };
  auto lo_empty = [&](int s) { return bar0 + 8u * (3 * R + s); };
  auto tfull_bar = [&](int s) { return bar0 + 8u * (3 * R + kLoStages + s); };
  auto tempty_bar = [&](int s) { return bar0 + 8u * (3 * R + kLoStages + 2 + s); };

  if (tid == 0) {
    for (int s = 0; s < R; ++s) { mbar_init(raw_full(s), p.use_tma ? 1 : 32); mbar_init(raw_empty(s), 1); mbar_init(conv_full(s), 32); }
    for (int s = 0; s < kLoStages; ++s) mbar_init(lo_empty(s), 1);
    for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 128); }
    fence_barrier_init();
  }
  if (warp == 4) tmem_alloc(smem_u32(tmem_slot), kTmemCols);

  // ---- stage this group's weights once: hi / lo split, canonical K-major layout (zero padded).
  // A task = one 16-byte piece of the layout (4 consecutive k of one output column); a thread keeps the 4 x kPieces
  // loads of its batch in flight, so the (L2-resident) weight fetch costs a few L2 round trips, not one per element.
  {
    const int pieces = (p.k_pad >> 2) * n_pad;
    constexpr int kPieces = 3;
    for (int e0 = tid; e0 < pieces; e0 += kTcThreads * kPieces) {
      float v[kPieces][4];
      uint32_t off[kPieces];
#pragma unroll
      for (int u = 0; u < kPieces; ++u) {
        const int e = e0 + u * kTcThreads;
        off[u] = 0xffffffffu;
#pragma unroll
        for (int j = 0; j < 4; ++j) v[u][j] = 0.f;
        if (e < pieces) {
          const int kq = e / n_pad, n = e - kq * n_pad;
          off[u] = static_cast<uint32_t>(kq) * lbo_b + static_cast<uint32_t>(n) * 16;
          const int ng = n_begin + n;
          if (n < n_count) {
            const int nb = ng >= p.n1 ? 1 : 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int k = 4 * kq + j;
              if (k < K) {
                const int kb = k >= p.k1 ? 1 : 0;
                const float* src = p.b[nb][kb];
                if (src != nullptr)
                  v[u][j] = __ldg(src + static_cast<int64_t>(ng - (nb ? p.n1 : 0)) * p.b_sn[nb][kb] +
                                  static_cast<int64_t>(k - (kb ? p.k1 : 0)) * p.b_sk[nb][kb]);
              }
            }
          }
        }
      }
#pragma unroll
      for (int u = 0; u < kPieces; ++u) {
        if (off[u] != 0xffffffffu) {
          const float4 hi = make_float4(tf32_hi(v[u][0]), tf32_hi(v[u][1]), tf32_hi(v[u][2]), tf32_hi(v[u][3]));
          *reinterpret_cast<float4*>(b_hi + off[u]) = hi;
          *reinterpret_cast<float4*>(b_lo + off[u]) = make_float4(v[u][0] - hi.x, v[u][1] - hi.y, v[u][2] - hi.z, v[u][3] - hi.w);
        }
      }
    }
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int n_chunks = p.k_pad / kChunkK;
  const int first_tile = blockIdx.x / p.n_split, tile_step = gridDim.x / p.n_split;
  const int my_tiles = first_tile < p.num_tiles ? (p.num_tiles - first_tile + tile_step - 1) / tile_step : 0;
  const int total_chunks = my_tiles * n_chunks;
  const uint32_t raw_addr = smem_u32(raw_ring), lo_addr = smem_u32(lo_ring);

  if (warp >= 9 && p.use_tma) {
    // ================= TMA producer: one lane, four [128 rows x 16 B] boxes per chunk =================
    // Each box is one 16-byte K piece of the 128 rows of the tile, which lands as 16 stacked core matrices - the
    // canonical no-swizzle K-major layout the MMA descriptors expect.  Rows past M and K pieces past the operand's
    // width are zero-filled by the TMA unit.
    if (warp == 9 && elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      int t = 0, j = 0;
      for (int c = 0; c < total_chunks; ++c) {
        const int row_base = (first_tile + t * tile_step) * kTileM;
        mbar_wait(raw_empty(stage), phase ^ 1u);
        mbar_arrive_expect_tx(raw_full(stage), kChunkBytes);
        const uint32_t dst = raw_addr + stage * kChunkBytes;
        if (p.use_tma == 2) {
          // one [128 rows x 16 floats] box in the 64-byte swizzle (k1 is a multiple of 16: a chunk never straddles A1 | A2)
          const int k = j * kChunkK;
          const bool second = k >= p.k1 && p.k2 > 0;
          tma_load_2d(dst, second ? &tm_a2 : &tm_a1, second ? k - p.k1 : k, row_base, raw_full(stage));
        } else {
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const int k = j * kChunkK + 4 * c4;
            const bool second = k >= p.k1 && p.k2 > 0;
            tma_load_2d(dst + c4 * (kTileM * 16), second ? &tm_a2 : &tm_a1, second ? k - p.k1 : k, row_base, raw_full(stage));
          }
        }
        if (++stage == R) { stage = 0; phase ^= 1u; }
        if (++j == n_chunks) { j = 0; ++t; }
      }
    }
  } else if (warp >= 9) {
    // ================= copy producers: each warp owns every other chunk =================
    const int pw = warp - 9;
    const int c4 = lane & 3, r0 = lane >> 2;                   // 16-byte K piece, first row (rows r0 + 8 i)
    int stage = pw % R;
    uint32_t phase = 0;
    int t = 0, j = pw;                                         // chunk -> (local tile, chunk in tile)
    while (j >= n_chunks) { j -= n_chunks; ++t; }
    for (int c = pw; c < total_chunks; c += kCopyWarps) {
      const int64_t row_base = static_cast<int64_t>(first_tile + t * tile_step) * kTileM;
      const int k = j * kChunkK + 4 * c4;
      const float* base;
      int64_t ld;
      if (k < p.k1) { base = p.a1 + k; ld = p.lda1; } else { base = p.a2 + (k - p.k1); ld = p.lda2; }
      const bool k_ok = k < K;
      mbar_wait(raw_empty(stage), phase ^ 1u);
      const uint32_t dst = raw_addr + stage * kChunkBytes + c4 * (kTileM * 16) + r0 * 16;
      if (p.ablate & 8) {
        mbar_arrive(raw_full(stage));
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int64_t row = row_base + r0 + 8 * i;
          const bool ok = k_ok && row < p.M;
          cp_async_16_zfill(dst + i * 128, ok ? base + row * ld : p.a1, ok ? 16u : 0u);
        }
        cp_async_mbar_arrive_noinc(raw_full(stage));
      }
      stage += kCopyWarps;
      if (stage >= R) { stage -= R; phase ^= 1u; }
      j += kCopyWarps;
      while (j >= n_chunks) { j -= n_chunks; ++t; }
    }
  } else if (warp >= 5) {
    // ================= converters: each warp owns every 4th chunk and one lo slot =================
    // kind::tf32 ignores the 13 low mantissa bits of its operands, so the raw chunk IS the hi operand:
    // only lo = a - (a & 0xffffe000) has to be produced.
    const int cw = warp - 5;
    int stage = cw % R;
    uint32_t phase = 0, lo_phase = 0;
    for (int c = cw; c < total_chunks; c += kConvWarps) {
      // When R is not a multiple of 4 the slot's previous chunk (c - R) belongs to another converter warp, and its copy may
      // still be in flight: raw_full would then be one phase behind, and a parity wait for this chunk would pass at once on
      // the completed phase of chunk c - 2R.  So first wait until the MMA has consumed chunk c - R (raw_empty cannot be a
      // phase ahead: chunk c is not consumed before it is converted).  The producer waits for the same before it copies
      // chunk c, so this never delays the conversion.
      mbar_wait(raw_empty(stage), phase ^ 1u);
      mbar_wait(raw_full(stage), phase);
      const uint32_t src = raw_addr + stage * kChunkBytes + lane * 16;
      float4 v[16];
      if (!(p.ablate & 1)) {
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = lds128(src + i * 512);
      }
      mbar_wait(lo_empty(cw), lo_phase ^ 1u);
      const uint32_t dlo = lo_addr + cw * kChunkBytes + lane * 16;
      if (!(p.ablate & 1))
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float4 l = make_float4(v[i].x - tf32_hi(v[i].x), v[i].y - tf32_hi(v[i].y), v[i].z - tf32_hi(v[i].z),
                                     v[i].w - tf32_hi(v[i].w));
        sts128(dlo + i * 512, l);
      }
      fence_proxy_async();
      mbar_arrive(conv_full(stage));
      stage += kConvWarps;
      if (stage >= R) { stage -= R; phase ^= 1u; }
      lo_phase ^= 1u;
    }
  } else if (warp == 4) {
    // ================= MMA issuer =================
    // The whole warp walks the loop converged (every operand below is warp-uniform, so the descriptors are
    // built in uniform registers); one elected lane issues the tcgen05 instructions.
    const uint32_t tmem_u = __shfl_sync(kFull, tmem_base, 0);
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(n_pad >> 3) << 17) |
                           (static_cast<uint32_t>(kTileM >> 4) << 24);
    constexpr uint32_t a_lbo = kTileM * 16, sbo = 128;
    // descriptors advance by adding (byte offset >> 4) to the 14-bit start-address field
    const bool sw64 = p.use_tma == 2;
    const uint64_t da_raw0 = sw64 ? make_desc_sw64(raw_addr) : make_desc(raw_addr, a_lbo, sbo);
    const uint64_t da_lo0 = sw64 ? make_desc_sw64(lo_addr) : make_desc(lo_addr, a_lbo, sbo);
    const uint32_t a_kstep = sw64 ? (32u >> 4) : ((2 * a_lbo) >> 4);      // second k-step of a chunk: +32 B inside the swizzle atom
    const uint64_t db_hi0 = make_desc(smem_u32(b_hi), lbo_b, sbo), db_lo0 = make_desc(smem_u32(b_lo), lbo_b, sbo);
    const uint32_t b_kstep = (2 * lbo_b) >> 4;
    const bool three = p.n_terms == 3;
    const bool leader = elect_one();              // the same lane issues every MMA and commit
    int stage = 0, lo = 0;
    uint32_t phase = 0;
    for (int t = 0; t < my_tiles; ++t) {
      const int acc = t & 1;
      mbar_wait(tempty_bar(acc), ((static_cast<uint32_t>(t) >> 1) & 1u) ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_u + static_cast<uint32_t>(acc) * 256u;
      for (int j = 0; j < n_chunks; ++j) {
        mbar_wait(conv_full(stage), phase);
        tc_fence_after();
        if (leader && (p.ablate & 4)) {
          umma_commit(raw_empty(stage));
          umma_commit(lo_empty(lo));
          if (j == n_chunks - 1) umma_commit(tfull_bar(acc));
        } else if (leader) {
          const uint64_t da_hi = da_raw0 + static_cast<uint32_t>(stage * (kChunkBytes >> 4));
          const uint64_t da_lo = da_lo0 + static_cast<uint32_t>(lo * (kChunkBytes >> 4));
          const uint64_t db_hi = db_hi0 + static_cast<uint32_t>(2 * j) * b_kstep;
          const uint64_t db_lo = db_lo0 + static_cast<uint32_t>(2 * j) * b_kstep;
#pragma unroll
          for (int s = 0; s < 2; ++s) {
            const uint32_t ao = s * a_kstep, bo = s * b_kstep;
            umma_tf32(d_tmem, da_hi + ao, db_hi + bo, idesc, (j | s) != 0 ? 1u : 0u);
            if (three) {
              umma_tf32(d_tmem, da_hi + ao, db_lo + bo, idesc, 1u);
              umma_tf32(d_tmem, da_lo + ao, db_hi + bo, idesc, 1u);
            }
          }
          umma_commit(raw_empty(stage));          // frees the raw (= hi) slot once these MMAs have read it
          umma_commit(lo_empty(lo));
          if (j == n_chunks - 1) umma_commit(tfull_bar(acc));   // accumulator complete -> epilogue
        }
        __syncwarp();
        if (++stage == R) { stage = 0; phase ^= 1u; }
        if (++lo == kLoStages) lo = 0;
      }
    }
  } else {
    // ================= epilogue: TMEM -> registers -> per-warp smem transpose -> coalesced global stores =====
    // tcgen05.ld gives one accumulator row per thread; storing that directly would touch 32 different 128-byte
    // lines per instruction.  Each warp bounces 32 rows x 32 columns through a padded staging tile so that
    // every store instruction writes 4 rows x 128 contiguous bytes.
    const uint32_t lane_base = static_cast<uint32_t>(warp * 32) << 16;
    const int n_end = n_begin + n_count;
    const uint32_t stage_addr = smem_u32(epi_stage) + warp * (32 * kEpiRowBytes);
    const int rr = lane >> 3, piece = lane & 7;                 // read-back geometry: 4 rows x 8 pieces per instruction
    for (int t = 0; t < my_tiles; ++t) {
      const int acc = t & 1;
      mbar_wait(tfull_bar(acc), (static_cast<uint32_t>(t) >> 1) & 1u);
      tc_fence_after();
      const int64_t row0 = static_cast<int64_t>(first_tile + t * tile_step) * kTileM + warp * 32;
      for (int col0 = 0; col0 < ((p.ablate & 2) ? 0 : n_pad); col0 += 32) {
        const int width = min(32, n_pad - col0);              // 16 or 32 columns in this block
        uint32_t r[32];
        {
          uint32_t (&ra)[16] = *reinterpret_cast<uint32_t (*)[16]>(&r[0]);
          uint32_t (&rb)[16] = *reinterpret_cast<uint32_t (*)[16]>(&r[16]);
          const uint32_t taddr = tmem_base + lane_base + static_cast<uint32_t>(acc) * 256u + static_cast<uint32_t>(col0);
          tmem_ld16(taddr, ra);
          if (width > 16) tmem_ld16(taddr + 16u, rb);
          tmem_ld_wait();
        }
        if (!BF16_C1 && p.use_tma_store) {
          // ---- TMA store: bias / sigmoid in registers, row `lane` into a 128B-swizzled [32 rows x 128 B] tile
          // (16-byte piece q of row r sits at piece q ^ (r & 7): conflict-free quarter-warp stores), one tensor store
          const int colg = n_begin + col0;                     // first output column of the block (multiple of 32)
          const bool to_c1 = colg < p.n1;
          const int cbase = to_c1 ? colg : colg - p.n1;
          const uint32_t tile = smem_u32(epi_stage) + warp * 4096;
          if (lane == 0) bulk_wait_read_all();                 // the previous block's tile has been read by the TMA unit
          __syncwarp();
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float4 v = make_float4(__uint_as_float(r[4 * q]), __uint_as_float(r[4 * q + 1]), __uint_as_float(r[4 * q + 2]),
                                   __uint_as_float(r[4 * q + 3]));
            if (4 * q >= width) v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (!to_c1) {
              if (p.bias2 != nullptr && cbase + 4 * q < p.n2) {
                const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias2 + cbase + 4 * q));
                v.x += bb.x; v.y += bb.y; v.z += bb.z; v.w += bb.w;
              }
              if (p.sigmoid2) {
                v.x = 1.f / (1.f + expf(-v.x)); v.y = 1.f / (1.f + expf(-v.y));
                v.z = 1.f / (1.f + expf(-v.z)); v.w = 1.f / (1.f + expf(-v.w));
              }
            }
            sts128(tile + lane * 128 + ((q ^ (lane & 7)) << 4), v);
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0 && !(p.ablate & 16)) {
            tma_store_2d(to_c1 ? &tm_c1 : &tm_c2, tile, cbase, static_cast<int>(row0));
            bulk_commit();
          }
          continue;
        }
        __syncwarp();                                          // previous block fully read back
#pragma unroll
        for (int q = 0; q < 8; ++q)
          if (4 * q < width)
            sts128(stage_addr + lane * kEpiRowBytes + q * 16,
                   make_float4(__uint_as_float(r[4 * q]), __uint_as_float(r[4 * q + 1]), __uint_as_float(r[4 * q + 2]),
                               __uint_as_float(r[4 * q + 3])));
        __syncwarp();
        const int col = n_begin + col0 + 4 * piece;
        if (4 * piece < width && col < n_end && !(p.ablate & 16)) {
          const bool to_c1 = col < p.n1;
          const int c2 = col - p.n1;
          float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
          if (!to_c1 && p.bias2 != nullptr) bb = __ldg(reinterpret_cast<const float4*>(p.bias2 + c2));
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int rl = 4 * i + rr;
            const int64_t row = row0 + rl;
            float4 v = lds128(stage_addr + rl * kEpiRowBytes + piece * 16);
            if (row < p.M) {
              if (to_c1) {
                if constexpr (BF16_C1) {
                  __stcs(reinterpret_cast<uint2*>(reinterpret_cast<bf16*>(p.c1) + row * p.ldc1 + col),
                         make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w)));
                } else {
                  __stcs(reinterpret_cast<float4*>(p.c1 + row * p.ldc1 + col), v);
                }
              } else {
                v.x += bb.x; v.y += bb.y; v.z += bb.z; v.w += bb.w;
                if (p.sigmoid2) {
                  v.x = 1.f / (1.f + expf(-v.x)); v.y = 1.f / (1.f + expf(-v.y));
                  v.z = 1.f / (1.f + expf(-v.z)); v.w = 1.f / (1.f + expf(-v.w));
                }
                __stcs(reinterpret_cast<float4*>(p.c2 + row * p.ldc2 + c2), v);
              }
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(tempty_bar(acc));
    }
    if (p.use_tma_store && lane == 0) bulk_wait_all();       // every tensor store has left shared memory and completed
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, kTmemCols);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static int round16(int v) { return (v + 15) / 16 * 16; }

struct TcPlan { int n_split, cols_per_group, raw_stages; size_t smem; };

// smallest column split that leaves a deep A ring next to the resident weights
static bool tc_plan(int k, int n, TcPlan& out) {
  const int k_pad = round16(k);
  const size_t fixed = static_cast<size_t>(kLoStages) * kChunkBytes + kEpiStageBytes + (3 * kMaxRawStages + kLoStages + 4) * 8 + 64;
  TcPlan best{0, 0, 0, 0};
  for (int s = 1; s <= 4; ++s) {
    const int cpg = round16(ceil_div(n, s));
    if (cpg < 16 || cpg > 256) continue;
    const size_t b_bytes = static_cast<size_t>(2) * cpg * k_pad * 4;
    if (b_bytes + fixed + 2 * kChunkBytes > static_cast<size_t>(kMaxSmem)) continue;
    int r = static_cast<int>(std::min<size_t>(kMaxRawStages, (kMaxSmem - b_bytes - fixed) / kChunkBytes));
    if (const char* cap = getenv("EGC_TC_MAX_RAW_STAGES")) r = std::max(kConvWarps, std::min(r, atoi(cap)));   // diagnostics
    if (r > best.raw_stages) best = TcPlan{s, cpg, r, b_bytes + fixed + static_cast<size_t>(r) * kChunkBytes};
    if (r >= 8) break;
  }
  out = best;
  return best.raw_stages >= kConvWarps;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

bool tc_aligned(const void* a, const void* b, const void* c, const void* d) {
  return aligned16(a) && aligned16(b) && aligned16(c) && aligned16(d);
}

bool project_tc_supported(int n, int f_in, int bd, int hab) {
  if (n < 1 || f_in % 4 || bd % 4 || hab % 4) return false;
  TcPlan a, b;
  return tc_plan(f_in, bd + hab, a) && tc_plan(bd + hab, f_in, b);
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
      f = nullptr;
    return reinterpret_cast<EncodeTiledFn>(f);
  }();
  return fn;
}
// [M rows x n floats] row-major output, 128B-swizzled boxes of 32 rows x 32 floats
static bool make_c_map(CUtensorMap* m, const float* base, int n, int64_t ld, int M) {
  EncodeTiledFn fn = encode_tiled();
  if (fn == nullptr || base == nullptr || n <= 0) return false;
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(n), static_cast<cuuint64_t>(M)};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 4};
  const cuuint32_t box[2] = {32, 32};
  const cuuint32_t es[2] = {1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// [M rows x k floats] row-major operand, boxes of 128 rows x 4 floats
static bool make_a_map(CUtensorMap* m, const float* base, int k, int64_t ld, int M) {
  EncodeTiledFn fn = encode_tiled();
  if (fn == nullptr || base == nullptr || k <= 0) return false;
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(k), static_cast<cuuint64_t>(M)};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 4};
  const cuuint32_t box[2] = {4, static_cast<cuuint32_t>(kTileM)};
  const cuuint32_t es[2] = {1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// [M rows x k floats] row-major operand, boxes of 128 rows x 16 floats in the 64-byte swizzle
static bool make_a_map_sw64(CUtensorMap* m, const float* base, int k, int64_t ld, int M) {
  EncodeTiledFn fn = encode_tiled();
  if (fn == nullptr || base == nullptr || k <= 0) return false;
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(k), static_cast<cuuint64_t>(M)};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * 4};
  const cuuint32_t box[2] = {static_cast<cuuint32_t>(kChunkK), static_cast<cuuint32_t>(kTileM)};
  const cuuint32_t es[2] = {1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <bool BF16_C1 = false>
static int launch_tc(TcParams& p, cudaStream_t st) {
  const int K = p.k1 + p.k2, N = p.n1 + p.n2;
  TcPlan plan;
  EGC_REQUIRE(tc_plan(K, N, plan), "tensor-core projection: shape does not fit shared memory");
  p.k_pad = round16(K);
  p.n_split = plan.n_split;
  p.cols_per_group = plan.cols_per_group;
  p.raw_stages = plan.raw_stages;
  p.num_tiles = ceil_div(p.M, kTileM);
  if (const char* ab = getenv("EGC_TC_ABLATE")) p.ablate = atoi(ab);
  static bool attr_set[kMaxDevices] = {};
  EGC_CUDA(max_dynamic_smem_once(reinterpret_cast<const void*>(k_project_tc<BF16_C1>), kMaxSmem, attr_set));
  // TMA feed of the A operand (default; EGC_TC_NO_TMA=1 keeps the cp.async producers): needs the driver's tensor-map
  // encoder and 16-byte aligned rows.  Measured on B200: arxiv shape 0.106 -> 0.088 ms, mag shape 0.217 -> 0.159 ms.
  alignas(64) CUtensorMap tm1, tm2;
  memset(&tm1, 0, sizeof(tm1));
  memset(&tm2, 0, sizeof(tm2));
  static const bool want_tma = getenv("EGC_TC_NO_TMA") == nullptr;
  p.use_tma = 0;
  // 64-byte swizzled boxes (default; EGC_TC_NO_SWIZZLE=1 keeps the four 16-byte boxes per chunk): one request per row and
  // chunk instead of four.  A chunk of 16 floats must not straddle the A1 | A2 boundary.
  static const bool want_sw64 = getenv("EGC_TC_NO_SWIZZLE") == nullptr;
  const bool tma_ok = want_tma && p.k1 % 4 == 0 && p.lda1 % 4 == 0 && (p.k2 == 0 || (p.k2 % 4 == 0 && p.lda2 % 4 == 0));
  if (tma_ok && want_sw64 && (p.k2 == 0 || p.k1 % kChunkK == 0) && make_a_map_sw64(&tm1, p.a1, p.k1, p.lda1, p.M) &&
      (p.k2 == 0 || make_a_map_sw64(&tm2, p.a2, p.k2, p.lda2, p.M)))
    p.use_tma = 2;
  else if (tma_ok && make_a_map(&tm1, p.a1, p.k1, p.lda1, p.M) && (p.k2 == 0 || make_a_map(&tm2, p.a2, p.k2, p.lda2, p.M)))
    p.use_tma = 1;
  // TMA tensor stores of the output (EGC_TC_TMA_STORE=1; experimental): column blocks of 32 must not straddle c1 | c2
  alignas(64) CUtensorMap tc1, tc2;
  memset(&tc1, 0, sizeof(tc1));
  memset(&tc2, 0, sizeof(tc2));
  static const bool want_tma_store = getenv("EGC_TC_TMA_STORE") != nullptr;
  p.use_tma_store = 0;
  if (!BF16_C1 && want_tma_store && p.n1 % 32 == 0 && p.cols_per_group % 32 == 0 && p.ldc1 % 4 == 0 && (p.n2 == 0 || (p.ldc2 % 4 == 0 && p.n2 % 4 == 0)) &&
      make_c_map(&tc1, p.c1, p.n1, p.ldc1, p.M) && (p.n2 == 0 || make_c_map(&tc2, p.c2, p.n2, p.ldc2, p.M)))
    p.use_tma_store = 1;
  const int per_group = std::max(1, std::min(p.num_tiles, sm_count() / p.n_split));
  const int grid = per_group * p.n_split;
  {
    LaunchScope ls("k_project_tc", st);
    k_project_tc<BF16_C1><<<grid, kTcThreads, plan.smem, st>>>(p, tm1, tm2, tc1, tc2);
  }
  EGC_LAUNCH_CHECK("k_project_tc");
  return EGC_OK;
}

int project_fwd_tc(const float* x, const float* w_bases, const float* w_comb, const float* b_comb, int n, int f_in,
                   int bd, int hab, int sigmoid, float* bases, float* weightings, int n_terms, cudaStream_t st) {
  EGC_REQUIRE(aligned16(x) && aligned16(bases) && aligned16(weightings) && (b_comb == nullptr || aligned16(b_comb)),
              "tensor-core projection needs 16-byte aligned tensors");
  TcParams p{};
  p.a1 = x; p.lda1 = f_in; p.k1 = f_in; p.a2 = nullptr; p.lda2 = 0; p.k2 = 0; p.M = n;
  p.b[0][0] = w_bases; p.b_sn[0][0] = 1; p.b_sk[0][0] = bd;          // B(n,k) = W_b[k][n]
  p.b[1][0] = w_comb; p.b_sn[1][0] = f_in; p.b_sk[1][0] = 1;         // B(n,k) = W_c[n][k]
  p.n1 = bd; p.n2 = hab;
  p.c1 = bases; p.ldc1 = bd; p.c2 = weightings; p.ldc2 = hab; p.bias2 = b_comb; p.sigmoid2 = sigmoid;
  p.n_terms = n_terms;
  return launch_tc(p, st);
}

int project_fwd_tc_bf16(const float* x, const float* w_bases, const float* w_comb, const float* b_comb, int n, int f_in,
                        int bd, int hab, int sigmoid, uint16_t* bases, float* weightings, int n_terms, cudaStream_t st) {
  EGC_REQUIRE(aligned16(x) && aligned16(bases) && aligned16(weightings) && (b_comb == nullptr || aligned16(b_comb)),
              "tensor-core projection needs 16-byte aligned tensors");
  TcParams p{};
  p.a1 = x; p.lda1 = f_in; p.k1 = f_in; p.a2 = nullptr; p.lda2 = 0; p.k2 = 0; p.M = n;
  p.b[0][0] = w_bases; p.b_sn[0][0] = 1; p.b_sk[0][0] = bd;
  p.b[1][0] = w_comb; p.b_sn[1][0] = f_in; p.b_sk[1][0] = 1;
  p.n1 = bd; p.n2 = hab;
  p.c1 = reinterpret_cast<float*>(bases); p.ldc1 = bd; p.c2 = weightings; p.ldc2 = hab; p.bias2 = b_comb; p.sigmoid2 = sigmoid;
  p.n_terms = n_terms;
  return launch_tc<true>(p, st);
}

size_t project_bwd_tc_workspace(int n, int f_in, int bd, int hab) {
  const size_t wg = std::max(wgrad_tc_workspace(n, f_in, bd, hab), wgrad_mn_workspace(n, f_in, bd, hab));
  return std::max(project_bwd_simt_workspace(n, f_in, bd, hab), wg + project_bwd_simt_workspace(n, f_in, bd, hab));
}

int project_bwd_tc(const float* x, const float* w_bases, const float* w_comb, const float* d_bases, const float* d_lin,
                   int n, int f_in, int bd, int hab, float* d_x, float* d_w_bases, float* d_w_comb, float* d_b_comb,
                   int n_terms, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  // d_x from unaligned tensors: the FFMA kernel below (egc_project_bwd refuses this for a forced tensor-core algorithm)
  float* d_x_simt = d_x != nullptr && !tc_aligned(d_bases, d_lin, d_x) ? d_x : nullptr;
  if (d_x != nullptr && d_x_simt == nullptr) {
    TcParams p{};
    p.a1 = d_bases; p.lda1 = bd; p.k1 = bd; p.a2 = d_lin; p.lda2 = hab; p.k2 = hab; p.M = n;
    p.b[0][0] = w_bases; p.b_sn[0][0] = bd; p.b_sk[0][0] = 1;         // k < bd : B(n,k) = W_b[n][k]
    p.b[0][1] = w_comb; p.b_sn[0][1] = 1; p.b_sk[0][1] = f_in;        // k >= bd: B(n,k) = W_c[k-bd][n]
    p.n1 = f_in; p.n2 = 0;
    p.c1 = d_x; p.ldc1 = f_in; p.c2 = nullptr; p.ldc2 = 0; p.bias2 = nullptr; p.sigmoid2 = 0;
    p.n_terms = n_terms;
    if (int rc = launch_tc(p, st)) return rc;
  }
  // parameter gradients: contraction over the node dimension (MN-major operands straight from TMA when the shape allows,
  // else the transposing kernel)
  const bool wg_ok = (d_w_bases != nullptr || d_w_comb != nullptr) && aligned16(x) && aligned16(d_bases) && aligned16(d_lin);
  if (wg_ok && wgrad_mn_supported(n, f_in, bd, hab)) {
    const size_t wg_bytes = std::max(wgrad_tc_workspace(n, f_in, bd, hab), wgrad_mn_workspace(n, f_in, bd, hab));
    if (int rc = wgrad_mn(x, d_bases, d_lin, n, f_in, bd, hab, d_w_bases, d_w_comb, n_terms, workspace, wg_bytes, st)) return rc;
    d_w_bases = nullptr;
    d_w_comb = nullptr;
    workspace = static_cast<char*>(workspace) + wg_bytes;
    workspace_bytes -= wg_bytes;
  } else if (wg_ok && wgrad_tc_supported(n, f_in, bd, hab)) {
    const size_t wg_bytes = std::max(wgrad_tc_workspace(n, f_in, bd, hab), wgrad_mn_workspace(n, f_in, bd, hab));
    if (int rc = wgrad_tc(x, d_bases, d_lin, n, f_in, bd, hab, d_w_bases, d_w_comb, n_terms, workspace, wg_bytes, st)) return rc;
    d_w_bases = nullptr;
    d_w_comb = nullptr;
    workspace = static_cast<char*>(workspace) + wg_bytes;
    workspace_bytes -= wg_bytes;
  }
  return project_bwd_simt(x, w_bases, w_comb, d_bases, d_lin, n, f_in, bd, hab, d_x_simt, d_w_bases, d_w_comb, d_b_comb,
                          workspace, workspace_bytes, st);
}

}  // namespace egc
