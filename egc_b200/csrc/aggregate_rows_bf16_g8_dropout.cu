// Instantiates the G = 8 family of the row-block forward aggregation kernel (aggregate_rows.cuh) with bf16 basis rows
// with DROP = true: the fused dropout after the ReLU (egc_dropout), in its own translation unit so that it compiles in
// parallel with the kernels without dropout.
#include <algorithm>

#include "aggregate_rows.cuh"

namespace egc {
int launch_aggregate_rows_bf16_g8_dropout(const AggParams& p, int mask, bool arg, int* task_counter, cudaStream_t st) {
  return launch_rows_family<8, bf16, true>(p, mask, arg, task_counter, st);
}
}  // namespace egc
