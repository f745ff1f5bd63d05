// Bounded Levenberg-Marquardt on the exact cost Hessian (invert.cu): the per-point device kernels of gpe_bank_solve and
// the compaction of the active list.  The host loop that drives them lives in gpemu.cu (DESIGN 4.6d).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace gpe {

// Per-point solver state: x (D) | g (D) | xt (D) | H (D, D) | f, pred, lambda, nu | (status, evaluations) as 2 x int32.
__host__ __device__ inline int64_t lm_state_doubles(int D) { return (int64_t)D * D + 3 * D + 5; }

struct LmProblem {
    int D;
    const double* lower;       // (D) or NULL (-inf)
    const double* upper;       // (D) or NULL (+inf)
    const double* prior_mean;  // rows of prior_ld doubles (0: one shared row) or NULL (0)
    int64_t prior_ld;
    const double* prior_prec;  // (D, D) or NULL (no prior)
    int max_iter;
    double ftol, xtol, gtol, lambda0;
};

// x0 (n, D) clipped into the box -> the state's x and the first evaluation rows xe (n, D); list = 0 .. n-1.
cudaError_t lm_init(const LmProblem& pb, const double* x0, int64_t n, double* state, double* xe, int* list, cudaStream_t st);
// One LM step for the n active points list[0 .. n): evaluation i (f, g, H without the prior) -> state of point list[i];
// flag[i] = 1 where the point stays active (its next trial point is in the state's xt).  first: the evaluation at x.
cudaError_t lm_step(const LmProblem& pb, int64_t n, const int* list, const double* fe, const double* ge, const double* he,
                    double* state, int* flag, bool first, cudaStream_t st);
// list_out = the entries of list whose flag is set, in order; *count their number.  temp: lm_select_temp(n) bytes.
size_t lm_select_temp(int64_t n);
cudaError_t lm_select(const int* list, const int* flag, int64_t n, int* list_out, int* count, void* temp, size_t temp_bytes,
                      cudaStream_t st);
// xe[i] = xt of point list[i]; with obs_ld > 0 also obs_out[i] (K) = obs row list[i].
cudaError_t lm_gather(const double* state, int D, const int* list, int64_t n, double* xe, const double* obs, int64_t obs_ld,
                      int64_t K, double* obs_out, cudaStream_t st);
// Outputs of n points from their state (any pointer but info may be NULL); cov = inv(H), NaN where H is not positive
// definite, symmetric bit for bit.
cudaError_t lm_output(int D, int64_t n, const double* state, double* x, double* cost, double* grad, double* hess, double* cov,
                      int32_t* info, cudaStream_t st);

}  // namespace gpe
