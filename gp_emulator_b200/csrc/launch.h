// Host-side launch helper and the per-DP kernel launchers (defined in predict_full_inst.cu, one object per DP).
#pragma once
#include <cuda_runtime.h>
#include <utility>
#include "host_common.h"
#include "predict_full.cuh"
#include "predict_mean.cuh"
#include "predict_bank_mean.cuh"
#include "predict_tiny.cuh"
#include "predict_tf32.cuh"
#include "predict_tf32_big.cuh"
#include "predict_var_large.cuh"

namespace gpe {

// Launch `kern` on `st` with `smem` bytes of dynamic shared memory and count the launch (gpe_launch_count).  The
// shared-memory opt-in is per function AND per device: it is set on every launch (microseconds) so that multi-device
// processes stay correct.
template <typename... P, typename... A>
cudaError_t launch_kernel(void (*kern)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, A&&... args) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<grid, block, smem, st>>>(std::forward<A>(args)...);
    count_launch();
    return cudaGetLastError();
}

// The kernels compiled for one padded input dimension DP.
struct DpKernels {
    int DP;
    cudaError_t (*full)(int cfg, const FullParams& p, int grid, size_t smem, cudaStream_t st);
    cudaError_t (*mean)(bool hess, const MeanParams& p, dim3 grid, size_t smem, cudaStream_t st);
    cudaError_t (*bank_mean)(int G, bool grad, const BankMeanParams& p, dim3 grid, size_t smem, cudaStream_t st);
    cudaError_t (*tiny)(const TinyParams& p, int grid, size_t smem, cudaStream_t st);
    // name of the fused instance `full` runs for (cfg, nt_act, symmetric); characters written, as snprintf
    int (*full_name)(int cfg, int nt_act, bool symmetric, char* buf, int len);
    // template name of the kernel `mean` runs for mean + gradient without the K* scratch
    const char* (*mean_name)();
};

#define GPE_DECL_DP(DPV) extern const DpKernels kKernelsDp##DPV;
GPE_DECL_DP(2)
GPE_DECL_DP(4)
GPE_DECL_DP(6)
GPE_DECL_DP(8)
GPE_DECL_DP(10)
GPE_DECL_DP(12)
GPE_DECL_DP(16)
GPE_DECL_DP(24)
GPE_DECL_DP(32)
#undef GPE_DECL_DP

// The kernels of the smallest compiled DP >= D (NULL: D > 32, no per-D compiled kernels).
inline const DpKernels* dp_kernels(int D) {
    static const DpKernels* const table[] = {&kKernelsDp2,  &kKernelsDp4,  &kKernelsDp6,  &kKernelsDp8, &kKernelsDp10,
                                             &kKernelsDp12, &kKernelsDp16, &kKernelsDp24, &kKernelsDp32};
    for (const DpKernels* k : table)
        if (k->DP >= D) return k;
    return nullptr;
}

cudaError_t launch_tf32(int DP, bool x3, const Tf32Params& p, int grid, size_t smem, cudaStream_t st);
cudaError_t launch_tf32_big(int DP, bool x3, const Tf32BigParams& p, int grid, size_t smem, cudaStream_t st);
cudaError_t launch_var_large(const VarLargeParams& p, int grid, size_t smem, cudaStream_t st);
// out (R, W) [+]= A (R, E <= 32) . basis, basis pre-tiled as [ks][Wp][4]; row r of A at (r / RD) ldn + (r % RD) ldd, element e
// at + e lde (project.cu)
cudaError_t project_rows(const double* A, int64_t R, int RD, int64_t ldn, int64_t lde, int64_t ldd, const double* b_tiled, int E,
                         int W, int Wp, double* out, int accumulate, cudaStream_t st);
// Forward cost of R rows (project.cu): cost (R) = 1/2 sum_w l_w (fwd - obs)^2 and, with grad, grad (R, D) of it, from the bank
// means mu (R, E) and gradients deriv (R, E, D); obs (R, obs_ld) or, obs_ld = 0, the shared observation in aux.
// aux (2 Wp) is filled by forward_cost_aux: weights (NULL: 1) and the shared observation (NULL: none), zero-padded to Wp.
cudaError_t forward_cost_aux(const double* weights, const double* obs1, int W, int Wp, double* aux, cudaStream_t st);
// s_out (R, E) or NULL: with it, s = (l o (fwd - obs)) . basis^T is stored too, and grad may be NULL.
cudaError_t forward_cost_rows(const double* mu, const double* deriv, int64_t R, int E, int D, const double* obs, int64_t obs_ld,
                              const double* aux, const double* b_tiled, int W, int Wp, int gy, double* part, double* cost,
                              double* grad, double* s_out, cudaStream_t st);
// C (E, E) = basis . diag(weights in aux) . basis^T, exactly symmetric.
cudaError_t forward_cost_curv(const double* b_tiled, const double* aux, int E, int Wp, double* C, cudaStream_t st);
size_t forward_cost_smem(int E);   // dynamic shared memory of forward_cost_rows for a bank of E emulators
// Column split gy of forward_cost_rows for a call of call_N points: > 1 (the column groups spread over gy CTAs per row tile,
// partial sums in part (gy, R, 1 + E)) when the row tiles alone leave most SMs idle.  A function of the call, not of a chunk.
int forward_cost_split(int64_t call_N, int W);
// group sizes the shared-difference bank kernel (predict_bank_mean.cuh) is compiled for: the G x (DP + 1) accumulators
// of a thread (G without the gradient) have to stay in registers
inline bool bank_group_ok(int DP, int G, bool grad) {
    if (!grad) return DP <= 16 && (G == 4 || G == 5 || G == 8 || G == 10);
    if (DP <= 10) return G >= 3 && G <= 5;
    if (DP == 12) return G == 3 || G == 4;
    if (DP == 16) return G == 2 || G == 3;
    return false;
}
static const int kTfDpList[] = {4, 8, 12, 16, 32};

}  // namespace gpe
