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
// dst[i] (K) = src row list[i], rows ld apart.
cudaError_t lm_gather_rows(const int* list, int64_t n, const double* src, int64_t ld, int64_t K, double* dst, cudaStream_t st);
// Outputs of n points from their state (any pointer but info may be NULL); cov = inv(H), NaN where H is not positive
// definite, symmetric bit for bit.
cudaError_t lm_output(int D, int64_t n, const double* state, double* x, double* cost, double* grad, double* hess, double* cov,
                      int32_t* info, cudaStream_t st);


// ---- time series (gpe_bank_solve_series, DESIGN 4.6g) ----
// The rows n = s T + t of a series keep the per-point state; the series' scalars live in those of its row s T.
struct LmSeries {
    int T;
    const double* coupling;    // (T - 1) or NULL (all 1)
    const double* R;           // (D, D) smoothness precision
    double* scratch;           // lm_series_scratch_doubles per series of the launch: the block factors L_t, M_t
};
__host__ __device__ inline int64_t lm_series_scratch_doubles(int D, int T) { return 2 * (int64_t)T * D * D; }
// One LM step for the n active series list[0 .. n): evaluation rows i T + t (f, g, H without prior and coupling) -> state
// of series list[i]; ge is overwritten.  flag[i] = 1 where the series stays active (trial rows in the state's xt).
cudaError_t lm_series_step(const LmProblem& pb, const LmSeries& sp, int64_t n, const int* list, const double* fe, double* ge,
                           const double* he, double* state, int* flag, bool first, cudaStream_t st);
// rows (n T) = the rows of the series list[0 .. n), in order.
cudaError_t lm_series_rows(const int* list, int64_t n, int T, int* rows, cudaStream_t st);
// Outputs of n series: x, grad (n T, D), hess and cov (n T, D, D) diagonal blocks, cost (n), info (n, 2); any but x and info
// may be NULL.  cov: NaN blocks where H is not positive definite, each block symmetric bit for bit.
cudaError_t lm_series_output(const LmProblem& pb, const LmSeries& sp, int64_t n, double* state, double* x, double* cost,
                             double* grad, double* hess, double* cov, int32_t* info, cudaStream_t st);

}  // namespace gpe
