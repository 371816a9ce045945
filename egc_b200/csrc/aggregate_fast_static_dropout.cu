// Instantiates the fast (warp-per-row) forward aggregation kernel for the specialised layer shapes
// with DROP = true: the fused dropout after the ReLU (egc_dropout), in its own translation unit so that it compiles in
// parallel with the kernels without dropout.
#include <algorithm>

#include "aggregate_fast.cuh"

namespace egc {
int launch_aggregate_fast_static_dropout(int cfg_index, const AggParams& p, bool arg, int smem_bytes, cudaStream_t st) {
  switch (cfg_index) {
#define X(I, ...) case I: return launch_fast_arg<StaticCfg<__VA_ARGS__>, true>(p, arg, smem_bytes, st);
    EGC_STATIC_CFGS(X)
#undef X
  }
  set_error("aggregate: unknown static configuration %d", cfg_index);
  return EGC_ERR_UNSUPPORTED;
}
}  // namespace egc
