// Bounded Levenberg-Marquardt on the exact cost Hessian, per point (gpe_bank_solve, DESIGN 4.6d): the damped, bounded
// Newton step, the compaction of the active list and the output pass.  One warp per point, D <= 32: lane r owns row r of
// the Hessian, which stays in registers with the gradient and the prior terms; the Cholesky factorisation is
// right-looking over shuffles.  Every sum runs in a fixed order over the lanes or the inputs and nothing is shared between
// points, so a point's result does not depend on its position in a launch.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <algorithm>

#include <cub/device/device_select.cuh>

#include "../../include/gpemu.h"
#include "host_common.h"
#include "invert.h"
#include "launch.h"

namespace gpe {

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kWarps = 4;                 // points per CTA
constexpr double kLambdaMax = 1e20;       // a Cholesky that still fails beyond this damping: stalled
constexpr double kScaleFloor = 1e-12;     // s_d = max(|H_dd|, kScaleFloor max_k |H_kk|) over the free set

// Sum over the lanes in a fixed tree, the result of lane 0 on every lane.
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(kFull, v, o);
    return __shfl_sync(kFull, v, 0);
}

// Maximum over the lanes; NaN if any lane holds NaN.
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double w = __shfl_xor_sync(kFull, v, o);
        v = (v != v || w != w) ? (v + w) : fmax(v, w);
    }
    return v;
}

// In place: lane r's row of a symmetric matrix (a[j], j < DP) -> row r of its lower Cholesky factor (a[j], j <= r).
// Returns false (on every lane) if a pivot is not positive.
template <int DP>
__device__ __forceinline__ bool chol(double (&a)[DP], int lane) {
    bool ok = true;
#pragma unroll
    for (int k = 0; k < DP; ++k) {
        const double piv = __shfl_sync(kFull, a[k], k);
        ok = ok && piv > 0.0;
        const double lkk = sqrt(piv);
        const double lrk = lane == k ? lkk : a[k] / lkk;
        if (lane >= k) a[k] = lrk;
#pragma unroll
        for (int j = 0; j < DP; ++j) {   // (j > k: a constant trip count, so that both loops unroll)
            if (j <= k) continue;
            const double ljk = __shfl_sync(kFull, lrk, j);
            if (lane >= j) a[j] = fma(-lrk, ljk, a[j]);
        }
    }
    return ok;
}

// Solve L L^T z = b with the factor of chol (lane r holds b_r, returns z_r).
template <int DP>
__device__ __forceinline__ double chol_solve(const double (&a)[DP], double b, int lane) {
#pragma unroll
    for (int k = 0; k < DP; ++k) {
        const double yk = __shfl_sync(kFull, b, k) / __shfl_sync(kFull, a[k], k);
        if (lane == k) b = yk;
        else if (lane > k) b = fma(-a[k], yk, b);
    }
#pragma unroll
    for (int k = DP - 1; k >= 0; --k) {
        const double zk = __shfl_sync(kFull, b, k) / __shfl_sync(kFull, a[k], k);
        if (lane == k) b = zk;
#pragma unroll
        for (int r = 0; r < DP; ++r) {
            if (r >= k) continue;
            const double lkr = __shfl_sync(kFull, a[r], k);
            if (lane == r) b = fma(-lkr, zk, b);
        }
    }
    return b;
}

struct StateView {
    double *x, *g, *xt, *H, *sc;
    int* info;
    __device__ StateView(double* base, int D)
        : x(base), g(base + D), xt(base + 2 * D), H(base + 3 * D), sc(base + 3 * D + D * D), info((int*)(sc + 4)) {}
};

// One LM step of active slot i (one warp).
template <int DP>
__device__ __forceinline__ void lm_step_point(const LmProblem& pb, int64_t i, const int* __restrict__ list,
                                              const double* __restrict__ fe, const double* __restrict__ ge,
                                              const double* __restrict__ he, double* __restrict__ state,
                                              int* __restrict__ flag, int first) {
    const int lane = threadIdx.x & 31;
    const int D = pb.D;
    const bool row = lane < D;
    const int64_t pt = list[i];
    StateView s(state + pt * lm_state_doubles(D), D);

    // the evaluation at slot i plus the prior: f and g_r here, row r of H when the point moves there
    double f = fe[i];
    double g = row ? ge[i * D + lane] : 0.0;
    const double xe = row ? (first ? s.x[lane] : s.xt[lane]) : 0.0;
    if (pb.prior_prec) {
        const double m = (row && pb.prior_mean) ? pb.prior_mean[pt * pb.prior_ld + lane] : 0.0;
        const double r = row ? xe - m : 0.0;
        double pr = 0.0;
#pragma unroll
        for (int j = 0; j < DP; ++j) {
            const double rj = __shfl_sync(kFull, r, j);
            if (row && j < D) pr = fma(pb.prior_prec[lane * D + j], rj, pr);
        }
        g += pr;
        f += 0.5 * warp_sum(r * pr);
    }

    double x, lam, nu;
    int nev, status = -1;
    bool moved = first != 0;
    if (first) {
        x = xe;
        lam = pb.lambda0;
        nu = 2.0;
        nev = 0;
        if (!isfinite(f)) status = GPE_SOLVE_NONFINITE;
    } else {
        x = row ? s.x[lane] : 0.0;
        const double f0 = s.sc[0], pred = s.sc[1];
        lam = s.sc[2];
        nu = s.sc[3];
        nev = s.info[1] + 1;
        const double rho = (f0 - f) / pred;
        if (f < f0 && rho > 0.0) {
            x = xe;
            const double t = 2.0 * rho - 1.0;
            lam *= fmax(1.0 / 3.0, 1.0 - t * t * t);
            nu = 2.0;
            moved = true;
            if (fabs(f0 - f) <= pb.ftol * fabs(f)) status = GPE_SOLVE_CONVERGED;
        } else {
            f = f0;
            g = row ? s.g[lane] : 0.0;
            lam *= nu;
            nu *= 2.0;
        }
    }
    // the state holds x, g, H of the point from here on (H is read back from it: one register row, not two)
    if (moved && row) {
        s.x[lane] = x;
        s.g[lane] = g;
        for (int j = 0; j < D; ++j)
            s.H[lane * D + j] = he[(i * D + lane) * D + j] + (pb.prior_prec ? pb.prior_prec[lane * D + j] : 0.0);
    }

    double pred = 0.0;
    if (status < 0) {
        const double lo = (row && pb.lower) ? pb.lower[lane] : -INFINITY;
        const double hi = (row && pb.upper) ? pb.upper[lane] : INFINITY;
        const bool free = row && !((x <= lo && g > 0.0) || (x >= hi && g < 0.0));
        if (warp_max(free ? fabs(g) : 0.0) <= pb.gtol) status = GPE_SOLVE_CONVERGED;
        else {
            const unsigned fmask = __ballot_sync(kFull, free);
            const double hd = row ? s.H[lane * D + lane] : 0.0;
            const double sd = fmax(fabs(hd), kScaleFloor * warp_max(free ? fabs(hd) : 0.0));
            double a[DP];
            for (;;) {   // (rejected steps raise lambda too: a step is only tried with lambda <= kLambdaMax)
                if (!(lam <= kLambdaMax)) { status = GPE_SOLVE_STALLED; break; }
#pragma unroll
                for (int j = 0; j < DP; ++j) {
                    const bool in = free && j < D && ((fmask >> j) & 1u);
                    const double hj = in ? s.H[lane * D + j] : 0.0;
                    a[j] = in ? (j == lane ? hj + lam * sd : hj) : (j == lane ? 1.0 : 0.0);
                }
                if (chol<DP>(a, lane)) break;
                lam *= nu;
                nu *= 2.0;
            }
            if (status < 0) {
                const double delta = chol_solve<DP>(a, free ? -g : 0.0, lane);
                const double xt = row ? fmin(fmax(x + delta, lo), hi) : 0.0;
                const double d = xt - x;
                if (warp_max(fabs(d)) <= pb.xtol * (warp_max(fabs(x)) + pb.xtol)) status = GPE_SOLVE_CONVERGED;
                else if (nev >= pb.max_iter) status = GPE_SOLVE_MAX_ITER;
                else {
                    double hdv = 0.0;
#pragma unroll
                    for (int j = 0; j < DP; ++j) {
                        const double dj = __shfl_sync(kFull, d, j);
                        if (row && j < D) hdv = fma(s.H[lane * D + j], dj, hdv);
                    }
                    pred = -(warp_sum(g * d) + 0.5 * warp_sum(d * hdv));
                    if (row) s.xt[lane] = xt;
                }
            }
        }
    }

    if (lane == 0) {
        s.sc[0] = f;
        s.sc[1] = pred;
        s.sc[2] = lam;
        s.sc[3] = nu;
        s.info[0] = status < 0 ? 0 : status;
        s.info[1] = nev;
        flag[i] = status < 0;
    }
}

// Warps stride over the active slots: any n is covered whatever the grid.
template <int DP>
__global__ void __launch_bounds__(32 * kWarps, 1) k_lm_step(LmProblem pb, int64_t n, const int* __restrict__ list,
                                                         const double* __restrict__ fe, const double* __restrict__ ge,
                                                         const double* __restrict__ he, double* __restrict__ state,
                                                         int* __restrict__ flag, int first) {
    for (int64_t i = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); i < n; i += (int64_t)gridDim.x * kWarps)
        lm_step_point<DP>(pb, i, list, fe, ge, he, state, flag, first);
}

__global__ void k_lm_init(LmProblem pb, const double* __restrict__ x0, int64_t n, double* __restrict__ state,
                          double* __restrict__ xe, int* __restrict__ list) {
    const int D = pb.D;
    const int64_t R = lm_state_doubles(D);
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n * D; k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p = k / D;
        const int d = (int)(k - p * D);
        double v = x0[k];
        if (pb.lower) v = fmax(v, pb.lower[d]);
        if (pb.upper) v = fmin(v, pb.upper[d]);
        state[p * R + d] = v;
        xe[k] = v;
        if (d == 0) list[p] = (int)p;
    }
}

__global__ void k_lm_gather(const double* __restrict__ state, int D, const int* __restrict__ list, int64_t n,
                            double* __restrict__ xe, const double* __restrict__ obs, int64_t obs_ld, int64_t K,
                            double* __restrict__ obs_out) {
    const int64_t R = lm_state_doubles(D), W = D + (obs_ld > 0 ? K : 0);
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n * W; k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = k / W, c = k - i * W;
        const int64_t p = list[i];
        if (c < D) xe[i * D + c] = state[p * R + 2 * D + c];
        else obs_out[i * K + (c - D)] = obs[p * obs_ld + (c - D)];
    }
}

// Outputs of point p (one warp).
template <int DP>
__device__ __forceinline__ void lm_output_point(int D, int64_t p, const double* __restrict__ state, double* __restrict__ x,
                                                double* __restrict__ cost, double* __restrict__ grad,
                                                double* __restrict__ hess, double* __restrict__ cov,
                                                int32_t* __restrict__ info) {
    const int lane = threadIdx.x & 31;
    const bool row = lane < D;
    StateView s(const_cast<double*>(state) + p * lm_state_doubles(D), D);
    if (row) {
        x[p * D + lane] = s.x[lane];
        if (grad) grad[p * D + lane] = s.g[lane];
        if (hess)
            for (int j = 0; j < D; ++j) hess[(p * D + lane) * D + j] = s.H[lane * D + j];
    }
    if (lane == 0) {
        if (cost) cost[p] = s.sc[0];
        info[2 * p] = s.info[0];
        info[2 * p + 1] = s.info[1];
    }
    if (!cov) return;
    double a[DP];
#pragma unroll
    for (int j = 0; j < DP; ++j) a[j] = (row && j < D) ? s.H[lane * D + j] : (j == lane ? 1.0 : 0.0);
    const bool ok = chol<DP>(a, lane);
    for (int c = 0; c < D; ++c) {
        const double z = ok ? chol_solve<DP>(a, lane == c ? 1.0 : 0.0, lane) : NAN;
        if (lane <= c) {
            cov[(p * D + lane) * D + c] = z;
            cov[(p * D + c) * D + lane] = z;
        }
    }
}

template <int DP>
__global__ void __launch_bounds__(32 * kWarps) k_lm_output(int D, int64_t n, const double* __restrict__ state,
                                                           double* __restrict__ x, double* __restrict__ cost,
                                                           double* __restrict__ grad, double* __restrict__ hess,
                                                           double* __restrict__ cov, int32_t* __restrict__ info) {
    for (int64_t p = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); p < n; p += (int64_t)gridDim.x * kWarps)
        lm_output_point<DP>(D, p, state, x, cost, grad, hess, cov, info);
}

// Blocks for `work` threads of `threads` a block; every kernel here strides, so the cap only bounds the grid.
unsigned grid_for(int64_t work, int threads) {
    return (unsigned)std::min<int64_t>((work + threads - 1) / threads, (int64_t)1 << 20);
}

}  // namespace

cudaError_t lm_init(const LmProblem& pb, const double* x0, int64_t n, double* state, double* xe, int* list, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    return launch_kernel(k_lm_init, grid_for(n * pb.D, 256), 256, 0, st, pb, x0, n, state, xe, list);
}

cudaError_t lm_step(const LmProblem& pb, int64_t n, const int* list, const double* fe, const double* ge, const double* he,
                    double* state, int* flag, bool first, cudaStream_t st) {
    auto k = pb.D <= 8 ? k_lm_step<8> : pb.D <= 16 ? k_lm_step<16> : k_lm_step<32>;
    if (n <= 0) return cudaSuccess;
    return launch_kernel(k, grid_for(n * 32, 32 * kWarps), 32 * kWarps, 0, st, pb, n, list, fe, ge, he, state, flag, (int)first);
}

size_t lm_select_temp(int64_t n) {
    size_t bytes = 0;
    cub::DeviceSelect::Flagged((void*)nullptr, bytes, (const int*)nullptr, (const int*)nullptr, (int*)nullptr, (int*)nullptr,
                               (int)n);
    return bytes;
}

cudaError_t lm_select(const int* list, const int* flag, int64_t n, int* list_out, int* count, void* temp, size_t temp_bytes,
                      cudaStream_t st) {
    count_launch();
    return cub::DeviceSelect::Flagged(temp, temp_bytes, list, flag, list_out, count, (int)n, st);
}

cudaError_t lm_gather(const double* state, int D, const int* list, int64_t n, double* xe, const double* obs, int64_t obs_ld,
                      int64_t K, double* obs_out, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    return launch_kernel(k_lm_gather, grid_for(n * (D + (obs_ld > 0 ? K : 0)), 256), 256, 0, st, state, D, list, n, xe, obs,
                         obs_ld, K, obs_out);
}

cudaError_t lm_output(int D, int64_t n, const double* state, double* x, double* cost, double* grad, double* hess, double* cov,
                      int32_t* info, cudaStream_t st) {
    auto k = D <= 8 ? k_lm_output<8> : D <= 16 ? k_lm_output<16> : k_lm_output<32>;
    if (n <= 0) return cudaSuccess;
    return launch_kernel(k, grid_for(n * 32, 32 * kWarps), 32 * kWarps, 0, st, D, n, state, x, cost, grad, hess, cov, info);
}

}  // namespace gpe
