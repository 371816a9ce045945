// Instantiates the G = 8 family of the row-block forward aggregation kernel (aggregate_rows.cuh) with bf16 basis rows
// for layer shapes without a specialised configuration.
#include <algorithm>

#include "aggregate_rows.cuh"

namespace egc {
int launch_aggregate_rows_bf16_g8(const AggParams& p, int mask, bool arg, int* task_counter, cudaStream_t st) {
  return launch_rows_family<8, bf16>(p, mask, arg, task_counter, st);
}
}  // namespace egc
