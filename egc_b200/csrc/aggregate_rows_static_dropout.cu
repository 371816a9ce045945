// Instantiates the row-block forward aggregation kernel (aggregate_rows.cuh) for the specialised layer shapes
// with DROP = true: the fused dropout after the ReLU (egc_dropout), in its own translation unit so that it compiles in
// parallel with the kernels without dropout.
#include <algorithm>

#include "aggregate_rows.cuh"

namespace egc {
int launch_aggregate_rows_static_dropout(int cfg_index, const AggParams& p, bool arg, int* task_counter, cudaStream_t st) {
  switch (cfg_index) {
#define X(I, ...) case I: return launch_rows_arg<StaticCfg<__VA_ARGS__>, float, true>(p, arg, task_counter, st);
    EGC_STATIC_CFGS(X)
#undef X
  }
  set_error("aggregate: unknown static configuration %d", cfg_index);
  return EGC_ERR_UNSUPPORTED;
}
}  // namespace egc
