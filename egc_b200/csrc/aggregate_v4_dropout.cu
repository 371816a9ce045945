// Instantiates the VEC=4 family of the general forward aggregation kernel (aggregate_impl.cuh)
// with DROP = true: the fused dropout after the ReLU (egc_dropout), in its own translation unit so that it compiles in
// parallel with the kernels without dropout.
#include "aggregate_impl.cuh"

namespace egc {
int launch_aggregate_v4_dropout(const AggParams& p, int mask, bool linw, bool arg, int smem_bytes, cudaStream_t st) {
  return launch_family<4, true>(p, mask, linw, arg, smem_bytes, st);
}
}  // namespace egc
