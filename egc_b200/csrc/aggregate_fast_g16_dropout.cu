// Instantiates the G = 16 family of the fast (warp-per-row) forward aggregation kernel
// with DROP = true: the fused dropout after the ReLU (egc_dropout), in its own translation unit so that it compiles in
// parallel with the kernels without dropout.
#include <algorithm>

#include "aggregate_fast.cuh"

namespace egc {
int launch_aggregate_fast_g16_dropout(const AggParams& p, int mask, bool arg, int smem_bytes, cudaStream_t st) {
  return launch_fast_family<16, true>(p, mask, arg, smem_bytes, st);
}
}  // namespace egc
