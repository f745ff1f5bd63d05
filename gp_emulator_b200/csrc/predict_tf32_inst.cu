// Instantiations of the tcgen05 / TMEM single-precision predict kernel (one per float4-padded input dimension).
#include "predict_tf32.cuh"
#include "predict_tf32_big.cuh"
#include "launch.h"

namespace gpe {

template <int DP, bool X3>
static cudaError_t launch_dp(const Tf32Params& p, int grid, size_t smem, cudaStream_t st) {
    return launch_kernel(k_predict_tf32<DP, X3>, grid, kTfThreads, smem, st, p);
}

cudaError_t launch_tf32(int DP, bool x3, const Tf32Params& p, int grid, size_t smem, cudaStream_t st) {
#define GPE_TF_CASE(DPV) \
    case DPV: return x3 ? launch_dp<DPV, true>(p, grid, smem, st) : launch_dp<DPV, false>(p, grid, smem, st);
    switch (DP) {
        GPE_TF_CASE(4)
        GPE_TF_CASE(8)
        GPE_TF_CASE(12)
        GPE_TF_CASE(16)
        GPE_TF_CASE(32)
        default: return cudaErrorInvalidValue;
    }
#undef GPE_TF_CASE
}

template <int DP, bool X3>
static cudaError_t launch_big_dp(const Tf32BigParams& p, int grid, size_t smem, cudaStream_t st) {
    return launch_kernel(k_predict_tf32_big<DP, X3>, grid, kTfThreads, smem, st, p);
}

cudaError_t launch_tf32_big(int DP, bool x3, const Tf32BigParams& p, int grid, size_t smem, cudaStream_t st) {
#define GPE_BIG_CASE(DPV) \
    case DPV: return x3 ? launch_big_dp<DPV, true>(p, grid, smem, st) : launch_big_dp<DPV, false>(p, grid, smem, st);
    switch (DP) {
        GPE_BIG_CASE(4)
        GPE_BIG_CASE(8)
        GPE_BIG_CASE(12)
        GPE_BIG_CASE(16)
        GPE_BIG_CASE(32)
        default: return cudaErrorInvalidValue;
    }
#undef GPE_BIG_CASE
}

}  // namespace gpe
