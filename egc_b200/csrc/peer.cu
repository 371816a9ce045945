// Row exchange of a row-partitioned graph over NVLink peer memory (one process per GPU).
//
// Every rank owns one "peer segment": device memory allocated here with cudaMalloc, exported as a CUDA IPC
// handle and mapped by the other ranks of the node.  All cross-GPU traffic of the layer is plain stores into a
// mapped segment issued by our own kernels (posted writes over NVLink - no round trips), ordered by epoch flags:
//
//   producer:  k_peer_push  (rows -> the consumer's segment)   ...kernel boundary...   k_peer_signal (flag = epoch)
//   consumer:  k_peer_wait  (spins on its OWN flags, local memory)                      then reads local memory
//
// The epoch lives in device memory and is advanced by a kernel, so a whole training step (pushes, signals, waits
// included) can be captured once in a CUDA graph and replayed.  The reference has no multi-GPU path; the contract
// is "same numbers as the single-GPU layer" (tests/test_gpu_dist.py).
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"

namespace egc {

// ---- data movers ----------------------------------------------------------------------------------
// One warp per row.  Segment s covers rows [seg_ptr[s], seg_ptr[s+1]) of the concatenated send list; row k of
// segment s is  src[s] + index[k] * width  (index == null: the k-th row of the segment, counted from its start)
// and lands at  dst[s] + (k - seg_ptr[s]) * width.  MAX_SEG: segment capacity of the parameter block - EGC_MAX_PEERS for
// one table per peer (EGConv), EGC_MAX_PUSH_SEGMENTS for one segment per (peer, node type) of a heterogeneous layer.
template <int MAX_SEG>
struct PushParams {
  const float* src[MAX_SEG];
  float* dst[MAX_SEG];
  int seg_ptr[MAX_SEG + 1];
  int n_seg;
  const int32_t* index;
  int width;
  // fused signal: the last CTA to finish raises flags[q][slot * world + rank] = *epoch for every slot of slot_mask
  uint32_t* flags[EGC_MAX_PEERS];
  int world, rank;
  uint32_t slot_mask;
  const uint32_t* epoch;
  unsigned int* counter;          // zero on entry, zero again on exit
};

// Thread `t` of the calling group raises the flags of peer t (q = t): the release stores are round trips over
// NVLink, so one thread per peer keeps them in flight together instead of paying world - 1 serial round trips.
__device__ __forceinline__ void raise_flags_of(uint32_t* const* flags, int world, int rank, uint32_t slot_mask, uint32_t e, int q) {
  if (q >= world || q == rank) return;
  for (int slot = 0; slot < 8; ++slot) {
    if (!((slot_mask >> slot) & 1u)) continue;
    uint32_t* f = flags[q] + slot * world + rank;
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(e) : "memory");
  }
}

// The segment of list row k: the last s < n_seg with seg_ptr[s] <= k (empty segments are skipped because their successor
// starts at the same row).  Up to EGC_MAX_PEERS segments an unrolled scan; beyond, a branchless binary search.
template <int MAX_SEG>
__device__ __forceinline__ int push_segment_of(const PushParams<MAX_SEG>& p, int k) {
  int s = 0;
  if constexpr (MAX_SEG <= EGC_MAX_PEERS) {
#pragma unroll
    for (int q = 1; q < MAX_SEG; ++q) s += (q < p.n_seg && k >= p.seg_ptr[q]) ? 1 : 0;
  } else {
#pragma unroll
    for (int step = MAX_SEG / 2; step > 0; step >>= 1) s += (s + step < p.n_seg && k >= p.seg_ptr[s + step]) ? step : 0;
  }
  return s;
}

template <int VEC, int MAX_SEG>
__global__ void __launch_bounds__(256) k_peer_push(const __grid_constant__ PushParams<MAX_SEG> p) {
  // A task = one VEC-float piece of one row; a thread keeps kPushUnroll pieces in flight (all loads, then all posted
  // stores), so narrow rows (256 B at the mag shape) use every lane and the copy runs at link speed instead of at the
  // latency of one  index -> row -> store  chain per warp.
  constexpr int kPushUnroll = 4;
  const int ppr = p.width / VEC;                                   // pieces per row
  const int64_t total = static_cast<int64_t>(p.seg_ptr[p.n_seg]) * ppr;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t t0 = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; t0 < total; t0 += stride * kPushUnroll) {
    float v[kPushUnroll][VEC];
    float* dst[kPushUnroll];
#pragma unroll
    for (int u = 0; u < kPushUnroll; ++u) {
      const int64_t t = t0 + u * stride;
      dst[u] = nullptr;
      if (t < total) {
        const int k = static_cast<int>(t / ppr), piece = static_cast<int>(t - static_cast<int64_t>(k) * ppr);
        const int s = push_segment_of(p, k);
        const int local = k - p.seg_ptr[s];
        const int64_t row = p.index != nullptr ? __ldg(p.index + k) : local;
        const float* src = p.src[s] + row * p.width + piece * VEC;
        dst[u] = p.dst[s] + static_cast<int64_t>(local) * p.width + piece * VEC;
        if constexpr (VEC == 4) {
          const float4 x = __ldg(reinterpret_cast<const float4*>(src));
          v[u][0] = x.x; v[u][1] = x.y; v[u][2] = x.z; v[u][3] = x.w;
        } else {
          v[u][0] = __ldg(src);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < kPushUnroll; ++u) {
      if (dst[u] != nullptr) {
        if constexpr (VEC == 4) *reinterpret_cast<float4*>(dst[u]) = make_float4(v[u][0], v[u][1], v[u][2], v[u][3]);
        else dst[u][0] = v[u][0];
      }
    }
  }
  if (p.slot_mask == 0u) return;
  // Fused signal: the CTA barrier orders every thread's posted stores before thread 0, whose system-scope fence is
  // cumulative over them (one fence per CTA instead of one per thread); the last CTA to count in raises the flags.
  __shared__ int s_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();
    const unsigned int prev = atomicAdd(p.counter, 1u);
    s_last = prev == gridDim.x - 1 ? 1 : 0;
    if (s_last) { __threadfence_system(); *p.counter = 0u; }
  }
  __syncthreads();
  if (s_last && threadIdx.x < EGC_MAX_PEERS) raise_flags_of(p.flags, p.world, p.rank, p.slot_mask, *p.epoch, threadIdx.x);
}

// ---- epoch flags ------------------------------------------------------------------------------------
// flags of a rank: uint32 [n_slots][world]; entry [slot][q] is written by rank q only.
__global__ void k_peer_epoch_advance(uint32_t* epoch) { *epoch += 1; }

struct SignalParams {
  uint32_t* flags[EGC_MAX_PEERS];   // every rank's flag array (mapped); own entry unused
  int world, rank;
  uint32_t slot_mask;
  const uint32_t* epoch;
};

__global__ void k_peer_signal(const __grid_constant__ SignalParams p) {
  __threadfence_system();
  raise_flags_of(p.flags, p.world, p.rank, p.slot_mask, *p.epoch, threadIdx.x);
}

// spins until every peer's entry of `slot` has reached epoch - lag; after `timeout_ns` it records the slot in *err and traps
__global__ void k_peer_wait(const uint32_t* flags, int world, int rank, int slot, uint32_t* epoch, uint32_t lag,
                            int advance, unsigned long long timeout_ns, uint32_t* err) {
  const int q = threadIdx.x;
  if (advance) {                               // a new step starts here: epoch += 1, then wait relative to it
    if (q == 0) *epoch += 1;
    __syncthreads();
  }
  if (q < world && q != rank) {
    const uint32_t e = *reinterpret_cast<volatile uint32_t*>(epoch);
    const uint32_t want = e > lag ? e - lag : 0u;
    const uint32_t* f = flags + slot * world + q;
    unsigned long long t0 = 0, now = 0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
      uint32_t v;
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
      if (static_cast<int32_t>(v - want) >= 0) break;
      __nanosleep(64);
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (now - t0 > timeout_ns) {
        // A peer never raised its flag: whatever this stream computes next would read stale or partial peer data.
        // Record which slot (readable through cudaMemcpy after the failure) and make the failure fatal: the trap
        // aborts the kernel, the stream and every later CUDA call of the process report an error.
        atomicExch(err, 1u + static_cast<uint32_t>(slot));
        __threadfence_system();
        __trap();
      }
    }
  }
  __syncthreads();
  __threadfence_system();
}

// ---- deterministic accumulation of what the peers pushed ----------------------------------------------
// One warp per local row that at least one peer contributed to: into[row] += sum over its entries (ascending
// peer order, fixed at plan time) of staging[entry].
template <int VEC>
__global__ void __launch_bounds__(256) k_peer_reduce_rows(const float* __restrict__ staging, const int32_t* __restrict__ rows,
                                                          const int32_t* __restrict__ ptr, const int32_t* __restrict__ entry,
                                                          int n_rows, int width, float* __restrict__ into) {
  const int ppr = width / VEC;
  const int64_t total = static_cast<int64_t>(n_rows) * ppr, stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; t < total; t += stride) {
    const int r = static_cast<int>(t / ppr), c = static_cast<int>(t - static_cast<int64_t>(r) * ppr) * VEC;
    float* dst = into + static_cast<int64_t>(__ldg(rows + r)) * width + c;
    const int b = __ldg(ptr + r), e = __ldg(ptr + r + 1);
    if constexpr (VEC == 4) {
      float4 acc = *reinterpret_cast<const float4*>(dst);
      for (int k = b; k < e; ++k) {                               // ascending peer order, fixed at plan time
        const float4 v = __ldcs(reinterpret_cast<const float4*>(staging + static_cast<int64_t>(__ldg(entry + k)) * width + c));
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      }
      *reinterpret_cast<float4*>(dst) = acc;
    } else {
      float acc = dst[0];
      for (int k = b; k < e; ++k) acc += __ldcs(staging + static_cast<int64_t>(__ldg(entry + k)) * width + c);
      dst[0] = acc;
    }
  }
}

// out[i] = slots[0][i] + slots[1][i] + ... in rank order (identical bits on every rank)
__global__ void k_peer_sum_slots(const float* __restrict__ slots, int world, int n, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float acc = 0.f;
  for (int q = 0; q < world; ++q) acc += __ldcs(slots + static_cast<int64_t>(q) * n + i);
  out[i] = acc;
}

// ---- one-shot all-reduce of a small replicated vector in ONE kernel ---------------------------------------
// (push my vector into slot [rank] of every rank -> flags -> wait for every peer's flag -> sum the slots in rank order).
// CTA c owns the float4 pieces c, c + gridDim.x, ...: it pushes them to every rank, and after the flags sums exactly
// those pieces, so its own slot needs no grid-wide ordering.  All CTAs must be co-resident (grid <= number of SMs).
struct AllReduceParams {
  const float* src;                  // [n] my contribution
  float* slot_of_me[EGC_MAX_PEERS];  // rank q's slot [rank] (mapped; q == rank: my own slots region)
  const float* my_slots;             // [world][n] what the peers pushed to me
  uint32_t* flags[EGC_MAX_PEERS];    // every rank's flag array (mapped)
  const uint32_t* my_flags;
  int world, rank, slot;
  const uint32_t* epoch;
  unsigned int* counter;             // zero on entry, zero again on exit
  int n;                             // multiple of 4
  float* out;                        // [n]
  unsigned long long timeout_ns;
  uint32_t* err;
};

__global__ void __launch_bounds__(256) k_peer_allreduce(const __grid_constant__ AllReduceParams p) {
  const int n4 = p.n >> 2;
  const int first = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
  for (int i = first; i < n4; i += stride) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p.src) + i);
    for (int q = 0; q < p.world; ++q) reinterpret_cast<float4*>(p.slot_of_me[q])[i] = v;
  }
  __shared__ int s_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();
    const unsigned int prev = atomicAdd(p.counter, 1u);
    s_last = prev == gridDim.x - 1 ? 1 : 0;
    if (s_last) { __threadfence_system(); *p.counter = 0u; }
  }
  __syncthreads();
  const uint32_t e = *p.epoch;
  if (s_last && threadIdx.x < EGC_MAX_PEERS) raise_flags_of(p.flags, p.world, p.rank, 1u << p.slot, e, threadIdx.x);
  const int q = threadIdx.x;
  if (q < p.world && q != p.rank) {
    const uint32_t* f = p.my_flags + p.slot * p.world + q;
    unsigned long long t0 = 0, now = 0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
      uint32_t v;
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
      if (static_cast<int32_t>(v - e) >= 0) break;
      __nanosleep(64);
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (now - t0 > p.timeout_ns) {
        atomicExch(p.err, 1u + static_cast<uint32_t>(p.slot));
        __threadfence_system();
        __trap();
      }
    }
  }
  __syncthreads();
  for (int i = first; i < n4; i += stride) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int r = 0; r < p.world; ++r) {                         // rank order: identical bits on every rank
      const float4 v = __ldcv(reinterpret_cast<const float4*>(p.my_slots + static_cast<int64_t>(r) * p.n) + i);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    reinterpret_cast<float4*>(p.out)[i] = acc;
  }
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

template <int MAX_SEG>
static int launch_peer_push(int32_t n_seg, const float* const* src, float* const* dst, const int32_t* seg_ptr,
                            const int32_t* index, int32_t width, uint32_t* const* flags, int32_t world, int32_t rank,
                            uint32_t slot_mask, const uint32_t* epoch, uint32_t* counter, void* stream) {
  PushParams<MAX_SEG> p{};
  bool vec = width % 4 == 0;
  p.n_seg = n_seg;
  for (int s = 0; s < n_seg; ++s) {
    p.src[s] = src[s];
    p.dst[s] = dst[s];
    p.seg_ptr[s] = seg_ptr[s];
    EGC_REQUIRE(seg_ptr[s + 1] >= seg_ptr[s], "egc_peer_push_rows: seg_ptr must be non-decreasing");
    if (seg_ptr[s + 1] > seg_ptr[s]) {
      EGC_REQUIRE(src[s] && dst[s], "egc_peer_push_rows: null segment pointer");
      vec = vec && aligned16(src[s]) && aligned16(dst[s]);
    }
  }
  for (int s = n_seg; s <= MAX_SEG; ++s) p.seg_ptr[s] = seg_ptr[n_seg];
  p.index = index;
  p.width = width;
  if (flags != nullptr && slot_mask != 0u && world > 1) {
    EGC_REQUIRE(world <= EGC_MAX_PEERS && rank >= 0 && rank < world && epoch && counter && slot_mask < 256u,
                "egc_peer_push_rows: bad signal arguments");
    for (int q = 0; q < world; ++q) p.flags[q] = flags[q];
    p.world = world; p.rank = rank; p.slot_mask = slot_mask; p.epoch = epoch; p.counter = counter;
  }
  const int total = seg_ptr[n_seg];
  cudaStream_t st = as_stream(stream);
  // one thread per 16-byte piece, 4 pieces in flight per thread (EGC_PEER_PUSH_CTAS_PER_SM: A/B runs; 1 CTA per SM measured
  // 10 % slower on the mag shape, profiles/r02d)
  static const int ctas_per_sm = [] { const char* e = getenv("EGC_PEER_PUSH_CTAS_PER_SM"); return e ? std::max(1, atoi(e)) : 8; }();
  const int64_t pieces = static_cast<int64_t>(total) * (vec ? width / 4 : width);
  const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((pieces + 1023) / 1024, static_cast<int64_t>(sm_count()) * ctas_per_sm)));
  {
    LaunchScope ls("k_peer_push", st);
    if (vec) k_peer_push<4, MAX_SEG><<<grid, 256, 0, st>>>(p);
    else k_peer_push<1, MAX_SEG><<<grid, 256, 0, st>>>(p);
  }
  EGC_LAUNCH_CHECK("k_peer_push");
  return EGC_OK;
}

}  // namespace egc

using namespace egc;

extern "C" {

int egc_peer_alloc(size_t bytes, void** ptr, egc_ipc_handle* handle) {
  EGC_REQUIRE(bytes > 0 && ptr && handle, "egc_peer_alloc: bad arguments");
  static_assert(sizeof(cudaIpcMemHandle_t) <= sizeof(egc_ipc_handle), "IPC handle does not fit");
  void* p = nullptr;
  EGC_CUDA(cudaMalloc(&p, bytes));
  EGC_CUDA(cudaMemset(p, 0, bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    set_error("cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
    return EGC_ERR_CUDA;
  }
  memset(handle, 0, sizeof(*handle));
  memcpy(handle, &h, sizeof(h));
  *ptr = p;
  return EGC_OK;
}

int egc_peer_free(void* ptr) {
  if (ptr != nullptr) EGC_CUDA(cudaFree(ptr));
  return EGC_OK;
}

int egc_peer_open(const egc_ipc_handle* handle, void** ptr) {
  EGC_REQUIRE(handle && ptr, "egc_peer_open: null pointer");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  EGC_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return EGC_OK;
}

int egc_peer_close(void* ptr) {
  if (ptr != nullptr) EGC_CUDA(cudaIpcCloseMemHandle(ptr));
  return EGC_OK;
}

int egc_peer_push_rows(int32_t n_seg, const float* const* src, float* const* dst, const int32_t* seg_ptr,
                       const int32_t* index, int32_t width, uint32_t* const* flags, int32_t world, int32_t rank,
                       uint32_t slot_mask, const uint32_t* epoch, uint32_t* counter, void* stream) {
  EGC_REQUIRE(n_seg >= 0 && n_seg <= EGC_MAX_PUSH_SEGMENTS && width > 0, "egc_peer_push_rows: n_seg=%d width=%d", n_seg, width);
  EGC_REQUIRE(seg_ptr && (n_seg == 0 || (src && dst)), "egc_peer_push_rows: null pointer");
  // up to one segment per peer (EGConv) the parameter block and the segment scan of the 8-entry kernel
  if (n_seg <= EGC_MAX_PEERS)
    return launch_peer_push<EGC_MAX_PEERS>(n_seg, src, dst, seg_ptr, index, width, flags, world, rank, slot_mask, epoch,
                                           counter, stream);
  return launch_peer_push<EGC_MAX_PUSH_SEGMENTS>(n_seg, src, dst, seg_ptr, index, width, flags, world, rank, slot_mask,
                                                 epoch, counter, stream);
}

int egc_peer_copy(void* dst, const void* src, size_t bytes, void* stream) {
  if (bytes == 0) return EGC_OK;
  EGC_REQUIRE(dst && src, "egc_peer_copy: null pointer");
  EGC_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, as_stream(stream)));   // copy engine: no SM is involved
  return EGC_OK;
}

int egc_peer_epoch_advance(uint32_t* epoch, void* stream) {
  EGC_REQUIRE(epoch, "egc_peer_epoch_advance: null pointer");
  cudaStream_t st = as_stream(stream);
  {
    LaunchScope ls("k_peer_epoch_advance", st);
    k_peer_epoch_advance<<<1, 1, 0, st>>>(epoch);
  }
  EGC_LAUNCH_CHECK("k_peer_epoch_advance");
  return EGC_OK;
}

int egc_peer_signal(uint32_t* const* flags, int32_t world, int32_t rank, uint32_t slot_mask, const uint32_t* epoch,
                    void* stream) {
  EGC_REQUIRE(flags && epoch && world >= 1 && world <= EGC_MAX_PEERS && rank >= 0 && rank < world && slot_mask < 256u,
              "egc_peer_signal: bad arguments");
  if (world == 1) return EGC_OK;
  SignalParams p{};
  for (int q = 0; q < world; ++q) p.flags[q] = flags[q];
  p.world = world; p.rank = rank; p.slot_mask = slot_mask; p.epoch = epoch;
  cudaStream_t st = as_stream(stream);
  {
    LaunchScope ls("k_peer_signal", st);
    k_peer_signal<<<1, 32, 0, st>>>(p);
  }
  EGC_LAUNCH_CHECK("k_peer_signal");
  return EGC_OK;
}

int egc_peer_wait(const uint32_t* my_flags, int32_t world, int32_t rank, int32_t slot, uint32_t* epoch,
                  uint32_t lag, int32_t advance, uint64_t timeout_ns, uint32_t* err, void* stream) {
  EGC_REQUIRE(my_flags && epoch && err && world >= 1 && world <= EGC_MAX_PEERS && rank >= 0 && rank < world && slot >= 0,
              "egc_peer_wait: bad arguments");
  if (world == 1 && !advance) return EGC_OK;
  cudaStream_t st = as_stream(stream);
  {
    LaunchScope ls("k_peer_wait", st);
    k_peer_wait<<<1, 32, 0, st>>>(my_flags, world, rank, slot, epoch, lag, advance, timeout_ns, err);
  }
  EGC_LAUNCH_CHECK("k_peer_wait");
  return EGC_OK;
}

int egc_peer_reduce_rows(const float* staging, const int32_t* rows, const int32_t* ptr, const int32_t* entry,
                         int32_t n_rows, int32_t width, float* into, void* stream) {
  EGC_REQUIRE(n_rows >= 0 && width > 0, "egc_peer_reduce_rows: n_rows=%d width=%d", n_rows, width);
  if (n_rows == 0) return EGC_OK;
  EGC_REQUIRE(staging && rows && ptr && entry && into, "egc_peer_reduce_rows: null pointer");
  cudaStream_t st = as_stream(stream);
  const bool vec = width % 4 == 0 && aligned16(staging) && aligned16(into);
  const int64_t pieces = static_cast<int64_t>(n_rows) * (vec ? width / 4 : width);
  const int grid = static_cast<int>(std::min<int64_t>((pieces + 255) / 256, static_cast<int64_t>(sm_count()) * 8));
  {
    LaunchScope ls("k_peer_reduce_rows", st);
    if (vec) k_peer_reduce_rows<4><<<grid, 256, 0, st>>>(staging, rows, ptr, entry, n_rows, width, into);
    else k_peer_reduce_rows<1><<<grid, 256, 0, st>>>(staging, rows, ptr, entry, n_rows, width, into);
  }
  EGC_LAUNCH_CHECK("k_peer_reduce_rows");
  return EGC_OK;
}

int egc_peer_allreduce(const float* src, float* const* slot_of_me, const float* my_slots, uint32_t* const* flags,
                       const uint32_t* my_flags, int32_t world, int32_t rank, int32_t slot, const uint32_t* epoch,
                       uint32_t* counter, int32_t n, float* out, uint64_t timeout_ns, uint32_t* err, void* stream) {
  EGC_REQUIRE(src && slot_of_me && my_slots && flags && my_flags && epoch && counter && out && err, "egc_peer_allreduce: null pointer");
  EGC_REQUIRE(world >= 1 && world <= EGC_MAX_PEERS && rank >= 0 && rank < world && slot >= 0 && slot < 8 && n >= 0 && n % 4 == 0,
              "egc_peer_allreduce: world=%d rank=%d slot=%d n=%d", world, rank, slot, n);
  if (n == 0) return EGC_OK;
  AllReduceParams p{};
  p.src = src; p.my_slots = my_slots; p.my_flags = my_flags; p.world = world; p.rank = rank; p.slot = slot;
  p.epoch = epoch; p.counter = counter; p.n = n; p.out = out; p.timeout_ns = timeout_ns; p.err = err;
  for (int q = 0; q < world; ++q) {
    EGC_REQUIRE(slot_of_me[q] && flags[q] && aligned16(slot_of_me[q]), "egc_peer_allreduce: bad mapped pointer of rank %d", q);
    p.slot_of_me[q] = slot_of_me[q];
    p.flags[q] = flags[q];
  }
  EGC_REQUIRE(aligned16(src) && aligned16(my_slots) && aligned16(out), "egc_peer_allreduce: buffers must be 16-byte aligned");
  cudaStream_t st = as_stream(stream);
  const int grid = std::max(1, std::min(ceil_div(n / 4, 256), std::min(sm_count(), 32)));   // co-resident by construction
  {
    LaunchScope ls("k_peer_allreduce", st);
    k_peer_allreduce<<<grid, 256, 0, st>>>(p);
  }
  EGC_LAUNCH_CHECK("k_peer_allreduce");
  return EGC_OK;
}

int egc_peer_sum_slots(const float* slots, int32_t world, int32_t n, float* out, void* stream) {
  EGC_REQUIRE(world >= 1 && n >= 0, "egc_peer_sum_slots: world=%d n=%d", world, n);
  if (n == 0) return EGC_OK;
  EGC_REQUIRE(slots && out, "egc_peer_sum_slots: null pointer");
  cudaStream_t st = as_stream(stream);
  {
    LaunchScope ls("k_peer_sum_slots", st);
    k_peer_sum_slots<<<ceil_div(n, 256), 256, 0, st>>>(slots, world, n, out);
  }
  EGC_LAUNCH_CHECK("k_peer_sum_slots");
  return EGC_OK;
}

}  // extern "C"
