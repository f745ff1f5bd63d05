// Instantiation + launcher of the M > 1024 variance kernel (predict_var_large.cuh).
#define GPE_VAR_LARGE_IMPL
#include "launch.h"

namespace gpe {

cudaError_t launch_var_large(const VarLargeParams& p, int grid, size_t smem, cudaStream_t st) {
    return launch_kernel(k_var_large, grid, kVlWarps * 32, smem, st, p);
}

}  // namespace gpe
