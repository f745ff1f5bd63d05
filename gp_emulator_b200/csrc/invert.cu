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

// Solve L y = b with the factor of chol (lane r holds b_r, returns y_r).
template <int DP>
__device__ __forceinline__ double tri_lower_solve(const double (&a)[DP], double b, int lane) {
#pragma unroll
    for (int k = 0; k < DP; ++k) {
        const double yk = __shfl_sync(kFull, b, k) / __shfl_sync(kFull, a[k], k);
        if (lane == k) b = yk;
        else if (lane > k) b = fma(-a[k], yk, b);
    }
    return b;
}

// Solve L^T z = b with the factor of chol (lane r holds b_r, returns z_r).
template <int DP>
__device__ __forceinline__ double tri_upper_solve(const double (&a)[DP], double b, int lane) {
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

// Solve L L^T z = b with the factor of chol (lane r holds b_r, returns z_r).
template <int DP>
__device__ __forceinline__ double chol_solve(const double (&a)[DP], double b, int lane) {
    return tri_upper_solve<DP>(a, tri_lower_solve<DP>(a, b, lane), lane);
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

// dst[i] (K) = src row list[i] (rows ld apart): the per-point weight rows and curvatures of the survivors (DESIGN 4.6f).
__global__ void k_lm_gather_rows(const int* __restrict__ list, int64_t n, const double* __restrict__ src, int64_t ld, int64_t K,
                                 double* __restrict__ dst) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n * K; k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = k / K, c = k - i * K;
        dst[k] = src[list[i] * ld + c];
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

// ---- time series (DESIGN 4.6g): the same LM per series of T dates, on the block-tridiagonal Hessian -----------------
// Row n = s T + t keeps the per-point state layout (x, g, xt, H = hess + P of date t); the series' f, pred, lambda, nu and
// info live in the scalars of its row s T.  The coupling adds c_t R to the diagonal blocks of dates t - 1 and t and
// -c_t R off the diagonal; terms whose c is 0 are skipped.  At T = 1 the step is k_lm_step's arithmetic, operation for
// operation (damp_diag), and the outputs are gpe_bank_solve_pw's bit for bit.

// Maximum of two values; NaN if either is NaN (the combination of warp_max).
__device__ __forceinline__ double max_nan(double v, double w) { return (v != v || w != w) ? (v + w) : fmax(v, w); }

// c_t of the pair (t - 1, t), 1 <= t < T.
__device__ __forceinline__ double series_c(const LmSeries& sp, int t) { return sp.coupling ? sp.coupling[t - 1] : 1.0; }

// c_t + c_{t+1}, with c_0 = c_T = 0: the coupling's weight of R in the diagonal block of date t.
__device__ __forceinline__ double series_cc(const LmSeries& sp, int t) {
    double cc = 0.0;
    if (t > 0) cc += series_c(sp, t);
    if (t + 1 < sp.T) cc += series_c(sp, t + 1);
    return cc;
}

// Entry (r, j) of the diagonal block of date t: H + cc R.
__device__ __forceinline__ double series_h(const double* __restrict__ H, const double* __restrict__ R, int D, int r, int j,
                                           double cc) {
    const double h = H[r * D + j];
    return cc != 0.0 ? fma(cc, R[r * D + j], h) : h;
}

// Lane r: (R v)_r, v_j on lane j.
template <int DP>
__device__ __forceinline__ double series_r_times(const double* __restrict__ R, int D, double v, int lane) {
    double acc = 0.0;
#pragma unroll
    for (int j = 0; j < DP; ++j) {
        const double vj = __shfl_sync(kFull, v, j);
        if (lane < D && j < D) acc = fma(R[lane * D + j], vj, acc);
    }
    return acc;
}

__device__ __forceinline__ bool series_free(const LmProblem& pb, const StateView& v, int lane) {
    if (lane >= pb.D) return false;
    const double x = v.x[lane], g = v.g[lane];
    const double lo = pb.lower ? pb.lower[lane] : -INFINITY;
    const double hi = pb.upper ? pb.upper[lane] : INFINITY;
    return !((x <= lo && g > 0.0) || (x >= hi && g < 0.0));
}

// Lane r: row r of a D x D block stored row-major, identity rows and columns beyond D.
template <int DP>
__device__ __forceinline__ void series_load(const double* __restrict__ blk, int D, int lane, double (&a)[DP]) {
#pragma unroll
    for (int j = 0; j < DP; ++j) a[j] = (lane < D && j < D) ? blk[lane * D + j] : (j == lane ? 1.0 : 0.0);
}

// hj + lambda s_j, rounded as k_lm_step<DP> rounds it: nvcc contracts it into one fma there at DP = 32 and keeps the product
// and the sum apart at DP = 8 and 16 (cuobjdump -sass).  Stated explicitly here, so that T = 1 is that kernel's arithmetic.
template <int DP>
__device__ __forceinline__ double damp_diag(double hj, double lam, double sd) {
    return DP == 32 ? fma(lam, sd, hj) : __dadd_rn(hj, __dmul_rn(lam, sd));
}

// Block Cholesky of the series' Hessian, right-looking over dates: C_t = A_t - M_t M_t^T, L_t = chol(C_t),
// M_{t+1} = B_{t+1} L_t^{-T}, L_t and M_t to the scratch (L: T blocks, then M: T blocks, M_0 unused).  damp: A_t and B_t
// are masked to the free set (identity rows and columns outside it) and A_t gets lambda diag(s), as in the point solver;
// otherwise the undamped H over all variables.  False (every lane) if a pivot is not positive.
template <int DP>
__device__ bool series_factor(const LmProblem& pb, const LmSeries& sp, double* __restrict__ st0, double* __restrict__ L,
                              double* __restrict__ M, bool damp, double lam, double hmax) {
    const int lane = threadIdx.x & 31;
    const int D = pb.D, T = sp.T;
    const bool row = lane < D;
    const int64_t RS = lm_state_doubles(D), DD = (int64_t)D * D;
    bool fr = damp ? series_free(pb, StateView(st0, D), lane) : row;
    for (int t = 0; t < T; ++t) {
        StateView v(st0 + t * RS, D);
        const unsigned fmask = __ballot_sync(kFull, fr);
        const double cc = series_cc(sp, t);
        double sd = 0.0;
        if (damp) {
            const double hd = row ? series_h(v.H, sp.R, D, lane, lane, cc) : 0.0;
            sd = fmax(fabs(hd), kScaleFloor * hmax);
        }
        double a[DP];
#pragma unroll
        for (int j = 0; j < DP; ++j) {
            const bool in = fr && j < D && ((fmask >> j) & 1u);
            const double hj = in ? series_h(v.H, sp.R, D, lane, j, cc) : 0.0;
            a[j] = in ? ((damp && j == lane) ? damp_diag<DP>(hj, lam, sd) : hj) : (j == lane ? 1.0 : 0.0);
        }
        if (t > 0 && series_c(sp, t) != 0.0) {
            const double* Mt = M + t * DD;
#pragma unroll
            for (int j = 0; j < DP; ++j) {
                if (!row || j >= D) continue;
                for (int k = 0; k < D; ++k) a[j] = fma(-Mt[lane * D + k], Mt[j * D + k], a[j]);
            }
        }
        if (!chol<DP>(a, lane)) return false;
        double* Lt = L + t * DD;
#pragma unroll
        for (int j = 0; j < DP; ++j)
            if (row && j < D) Lt[lane * D + j] = a[j];
        __syncwarp();
        if (t + 1 == T) break;
        const bool frn = damp ? series_free(pb, StateView(st0 + (t + 1) * RS, D), lane) : row;
        const double c = series_c(sp, t + 1);
        if (c != 0.0) {
            // row r of M_{t+1}: L_t m = b_r, b_r = -c R[r, :] on the free (t + 1, r) x (t, k) entries
            double m[DP];
#pragma unroll
            for (int k = 0; k < DP; ++k) {
                double acc = (frn && k < D && ((fmask >> k) & 1u)) ? -c * sp.R[lane * D + k] : 0.0;
#pragma unroll
                for (int j = 0; j < DP; ++j)
                    if (j < k && k < D) acc = fma(-Lt[k * D + j], m[j], acc);
                m[k] = k < D ? acc / Lt[k * D + k] : 0.0;
            }
            double* Mn = M + (t + 1) * DD;
#pragma unroll
            for (int k = 0; k < DP; ++k)
                if (row && k < D) Mn[lane * D + k] = m[k];
            __syncwarp();
        }
        fr = frn;
    }
    return true;
}

// One LM step of active series slot i (one warp): evaluation rows i T + t.  The evaluation's gradient rows (ge) are
// overwritten with the series' gradient, coupling included.
template <int DP>
__device__ __forceinline__ void lm_series_step_one(const LmProblem& pb, const LmSeries& sp, int64_t i,
                                                   const int* __restrict__ list, const double* __restrict__ fe,
                                                   double* __restrict__ ge, const double* __restrict__ he,
                                                   double* __restrict__ state, int* __restrict__ flag, int first) {
    const int lane = threadIdx.x & 31;
    const int D = pb.D, T = sp.T;
    const bool row = lane < D;
    const int64_t s = list[i], RS = lm_state_doubles(D), DD = (int64_t)D * D;
    double* st0 = state + s * T * RS;
    StateView s0(st0, D);
    double* L = sp.scratch + s * 2 * T * DD;
    double* M = L + T * DD;

    // 1. f of the series at the evaluated rows (prior and coupling included); the series' gradient replaces ge
    double f = 0.0, xprev = 0.0, gprev = 0.0;
    for (int t = 0; t < T; ++t) {
        const int64_t n = s * T + t, e = i * T + t;
        StateView v(st0 + t * RS, D);
        double ft = fe[e];
        double g = row ? ge[e * D + lane] : 0.0;
        const double xe = row ? (first ? v.x[lane] : v.xt[lane]) : 0.0;
        if (pb.prior_prec) {
            const double m = (row && pb.prior_mean) ? pb.prior_mean[n * pb.prior_ld + lane] : 0.0;
            const double r = row ? xe - m : 0.0;
            double pr = 0.0;
#pragma unroll
            for (int j = 0; j < DP; ++j) {
                const double rj = __shfl_sync(kFull, r, j);
                if (row && j < D) pr = fma(pb.prior_prec[lane * D + j], rj, pr);
            }
            g += pr;
            ft += 0.5 * warp_sum(r * pr);
        }
        f = t == 0 ? ft : f + ft;
        if (t > 0) {
            const double c = series_c(sp, t);
            if (c != 0.0) {
                const double dx = xe - xprev;
                const double rd = series_r_times<DP>(sp.R, D, dx, lane);
                f += 0.5 * (c * warp_sum(dx * rd));
                g = fma(c, rd, g);
                gprev = fma(-c, rd, gprev);
            }
            if (row) ge[(e - 1) * D + lane] = gprev;
        }
        xprev = xe;
        gprev = g;
    }
    if (row) ge[(i * T + T - 1) * D + lane] = gprev;

    // 2. accept or reject on the series' f (as the point solver)
    double lam, nu;
    int nev, status = -1;
    bool moved = first != 0;
    if (first) {
        lam = pb.lambda0;
        nu = 2.0;
        nev = 0;
        if (!isfinite(f)) status = GPE_SOLVE_NONFINITE;
    } else {
        const double f0 = s0.sc[0], pred = s0.sc[1];
        lam = s0.sc[2];
        nu = s0.sc[3];
        nev = s0.info[1] + 1;
        const double rho = (f0 - f) / pred;
        if (f < f0 && rho > 0.0) {
            const double t3 = 2.0 * rho - 1.0;
            lam *= fmax(1.0 / 3.0, 1.0 - t3 * t3 * t3);
            nu = 2.0;
            moved = true;
            if (fabs(f0 - f) <= pb.ftol * fabs(f)) status = GPE_SOLVE_CONVERGED;
        } else {
            f = f0;
            lam *= nu;
            nu *= 2.0;
        }
    }
    if (moved && row) {
        for (int t = 0; t < T; ++t) {
            const int64_t e = i * T + t;
            StateView v(st0 + t * RS, D);
            if (!first) v.x[lane] = v.xt[lane];
            v.g[lane] = ge[e * D + lane];
            for (int j = 0; j < D; ++j)
                v.H[lane * D + j] = he[(e * D + lane) * D + j] + (pb.prior_prec ? pb.prior_prec[lane * D + j] : 0.0);
        }
    }
    __syncwarp();

    double pred = 0.0;
    if (status < 0) {
        // 3. projected-gradient test and the scale floor, maxima over the series
        double gmax = 0.0, hmax = 0.0;
        for (int t = 0; t < T; ++t) {
            StateView v(st0 + t * RS, D);
            const bool fr = series_free(pb, v, lane);
            const double hd = row ? series_h(v.H, sp.R, D, lane, lane, series_cc(sp, t)) : 0.0;
            const double gm = warp_max(fr ? fabs(v.g[lane]) : 0.0), hm = warp_max(fr ? fabs(hd) : 0.0);
            gmax = t == 0 ? gm : max_nan(gmax, gm);
            hmax = t == 0 ? hm : max_nan(hmax, hm);
        }
        if (gmax <= pb.gtol) status = GPE_SOLVE_CONVERGED;
        else {
            for (;;) {
                if (!(lam <= kLambdaMax)) { status = GPE_SOLVE_STALLED; break; }
                if (series_factor<DP>(pb, sp, st0, L, M, true, lam, hmax)) break;
                lam *= nu;
                nu *= 2.0;
            }
        }
        if (status < 0) {
            // 4. forward then backward block substitution; the step goes through the rows' xt
            double a[DP];
            double y = 0.0;
            for (int t = 0; t < T; ++t) {
                StateView v(st0 + t * RS, D);
                double b = series_free(pb, v, lane) ? -v.g[lane] : 0.0;
                if (t > 0 && series_c(sp, t) != 0.0) {
                    const double* Mt = M + t * DD;
                    double acc = 0.0;
#pragma unroll
                    for (int k = 0; k < DP; ++k) {
                        const double yk = __shfl_sync(kFull, y, k);
                        if (row && k < D) acc = fma(Mt[lane * D + k], yk, acc);
                    }
                    b -= acc;
                }
                series_load<DP>(L + t * DD, D, lane, a);
                y = tri_lower_solve<DP>(a, b, lane);
                if (row) v.xt[lane] = y;
            }
            __syncwarp();
            double z = 0.0;
            for (int t = T - 1; t >= 0; --t) {
                StateView v(st0 + t * RS, D);
                double b = row ? v.xt[lane] : 0.0;
                if (t + 1 < T && series_c(sp, t + 1) != 0.0) {
                    const double* Mn = M + (t + 1) * DD;
                    double acc = 0.0;
#pragma unroll
                    for (int k = 0; k < DP; ++k) {
                        const double zk = __shfl_sync(kFull, z, k);
                        if (row && k < D) acc = fma(Mn[k * D + lane], zk, acc);
                    }
                    b -= acc;
                }
                series_load<DP>(L + t * DD, D, lane, a);
                z = tri_upper_solve<DP>(a, b, lane);
                if (row) v.xt[lane] = z;
            }
            __syncwarp();
            // 5. clip, the xtol test and the predicted reduction -(g^T d + 1/2 d^T H d)
            double maxd = 0.0, maxx = 0.0, gd = 0.0, q = 0.0, dprev = 0.0;
            for (int t = 0; t < T; ++t) {
                StateView v(st0 + t * RS, D);
                const double lo = (row && pb.lower) ? pb.lower[lane] : -INFINITY;
                const double hi = (row && pb.upper) ? pb.upper[lane] : INFINITY;
                const double x = row ? v.x[lane] : 0.0, g = row ? v.g[lane] : 0.0;
                const double xt = row ? fmin(fmax(x + v.xt[lane], lo), hi) : 0.0;
                const double d = xt - x;
                const double md = warp_max(fabs(d)), mx = warp_max(fabs(x));
                maxd = t == 0 ? md : max_nan(maxd, md);
                maxx = t == 0 ? mx : max_nan(maxx, mx);
                double hdv = 0.0;
#pragma unroll
                for (int j = 0; j < DP; ++j) {
                    const double dj = __shfl_sync(kFull, d, j);
                    if (row && j < D) hdv = fma(v.H[lane * D + j], dj, hdv);
                }
                const double gdt = warp_sum(g * d), qt = warp_sum(d * hdv);
                gd = t == 0 ? gdt : gd + gdt;
                q = t == 0 ? qt : q + qt;
                if (t > 0) {
                    const double c = series_c(sp, t);
                    if (c != 0.0) {
                        const double dd = d - dprev;
                        q += c * warp_sum(dd * series_r_times<DP>(sp.R, D, dd, lane));
                    }
                }
                if (row) v.xt[lane] = xt;
                dprev = d;
            }
            if (maxd <= pb.xtol * (maxx + pb.xtol)) status = GPE_SOLVE_CONVERGED;
            else if (nev >= pb.max_iter) status = GPE_SOLVE_MAX_ITER;
            else pred = -(gd + 0.5 * q);
        }
    }

    if (lane == 0) {
        s0.sc[0] = f;
        s0.sc[1] = pred;
        s0.sc[2] = lam;
        s0.sc[3] = nu;
        s0.info[0] = status < 0 ? 0 : status;
        s0.info[1] = nev;
        flag[i] = status < 0;
    }
}

template <int DP>
__global__ void __launch_bounds__(32 * kWarps, 1) k_lm_series_step(LmProblem pb, LmSeries sp, int64_t n,
                                                                const int* __restrict__ list, const double* __restrict__ fe,
                                                                double* __restrict__ ge, const double* __restrict__ he,
                                                                double* __restrict__ state, int* __restrict__ flag,
                                                                int first) {
    for (int64_t i = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); i < n; i += (int64_t)gridDim.x * kWarps)
        lm_series_step_one<DP>(pb, sp, i, list, fe, ge, he, state, flag, first);
}

// rows[i T + t] = list[i] T + t: the rows of the listed series, for the row gathers of the point solver.
__global__ void k_lm_series_rows(const int* __restrict__ list, int64_t n, int T, int* __restrict__ rows) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n * T; k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = k / T;
        rows[k] = (int)(list[i] * (int64_t)T + (k - i * T));
    }
}

// Outputs of series p (one warp).  cov: the diagonal blocks of inv(H) by Sigma_{T-1} = (L L^T)^{-1} and
// Sigma_t = L_t^{-T} (I + M_{t+1}^T Sigma_{t+1} M_{t+1}) L_t^{-1}, one column at a time, Sigma_{t+1} read back from cov.
template <int DP>
__device__ __forceinline__ void lm_series_output_one(const LmProblem& pb, const LmSeries& sp, int64_t p,
                                                     double* __restrict__ state, double* __restrict__ x,
                                                     double* __restrict__ cost, double* __restrict__ grad,
                                                     double* __restrict__ hess, double* __restrict__ cov,
                                                     int32_t* __restrict__ info) {
    const int lane = threadIdx.x & 31;
    const int D = pb.D, T = sp.T;
    const bool row = lane < D;
    const int64_t RS = lm_state_doubles(D), DD = (int64_t)D * D;
    double* st0 = state + p * T * RS;
    StateView s0(st0, D);
    for (int t = 0; t < T; ++t) {
        const int64_t n = p * T + t;
        StateView v(st0 + t * RS, D);
        if (!row) continue;
        x[n * D + lane] = v.x[lane];
        if (grad) grad[n * D + lane] = v.g[lane];
        if (hess) {
            const double cc = series_cc(sp, t);
            for (int j = 0; j < D; ++j) hess[(n * D + lane) * D + j] = series_h(v.H, sp.R, D, lane, j, cc);
        }
    }
    if (lane == 0) {
        if (cost) cost[p] = s0.sc[0];
        info[2 * p] = s0.info[0];
        info[2 * p + 1] = s0.info[1];
    }
    if (!cov) return;
    double* L = sp.scratch + p * 2 * T * DD;
    double* M = L + T * DD;
    const bool ok = series_factor<DP>(pb, sp, st0, L, M, false, 0.0, 0.0);
    double a[DP];
    for (int t = T - 1; t >= 0; --t) {
        const int64_t n = p * T + t;
        const bool next = t + 1 < T && series_c(sp, t + 1) != 0.0;
        const double* Mn = M + (t + 1) * DD;
        const double* Sn = cov + (n + 1) * DD;
        if (ok) series_load<DP>(L + t * DD, D, lane, a);
        for (int c = 0; c < D; ++c) {
            double z = NAN;
            if (ok) {
                double u = tri_lower_solve<DP>(a, lane == c ? 1.0 : 0.0, lane);
                if (next) {
                    double v = 0.0, w = 0.0, y = 0.0;
#pragma unroll
                    for (int k = 0; k < DP; ++k) {
                        const double uk = __shfl_sync(kFull, u, k);
                        if (row && k < D) v = fma(Mn[lane * D + k], uk, v);
                    }
#pragma unroll
                    for (int k = 0; k < DP; ++k) {
                        const double vk = __shfl_sync(kFull, v, k);
                        if (row && k < D) w = fma(Sn[lane * D + k], vk, w);
                    }
#pragma unroll
                    for (int k = 0; k < DP; ++k) {
                        const double wk = __shfl_sync(kFull, w, k);
                        if (row && k < D) y = fma(Mn[k * D + lane], wk, y);
                    }
                    u += y;
                }
                z = tri_upper_solve<DP>(a, u, lane);
            }
            if (lane <= c) {
                cov[(n * D + lane) * D + c] = z;
                cov[(n * D + c) * D + lane] = z;
            }
        }
        __syncwarp();
    }
}

template <int DP>
__global__ void __launch_bounds__(32 * kWarps, 1) k_lm_series_output(LmProblem pb, LmSeries sp, int64_t n, double* __restrict__ state,
                                                                  double* __restrict__ x, double* __restrict__ cost,
                                                                  double* __restrict__ grad, double* __restrict__ hess,
                                                                  double* __restrict__ cov, int32_t* __restrict__ info) {
    for (int64_t p = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); p < n; p += (int64_t)gridDim.x * kWarps)
        lm_series_output_one<DP>(pb, sp, p, state, x, cost, grad, hess, cov, info);
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

cudaError_t lm_gather_rows(const int* list, int64_t n, const double* src, int64_t ld, int64_t K, double* dst, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    return launch_kernel(k_lm_gather_rows, grid_for(n * K, 256), 256, 0, st, list, n, src, ld, K, dst);
}

cudaError_t lm_output(int D, int64_t n, const double* state, double* x, double* cost, double* grad, double* hess, double* cov,
                      int32_t* info, cudaStream_t st) {
    auto k = D <= 8 ? k_lm_output<8> : D <= 16 ? k_lm_output<16> : k_lm_output<32>;
    if (n <= 0) return cudaSuccess;
    return launch_kernel(k, grid_for(n * 32, 32 * kWarps), 32 * kWarps, 0, st, D, n, state, x, cost, grad, hess, cov, info);
}

cudaError_t lm_series_step(const LmProblem& pb, const LmSeries& sp, int64_t n, const int* list, const double* fe, double* ge,
                           const double* he, double* state, int* flag, bool first, cudaStream_t st) {
    auto k = pb.D <= 8 ? k_lm_series_step<8> : pb.D <= 16 ? k_lm_series_step<16> : k_lm_series_step<32>;
    if (n <= 0) return cudaSuccess;
    return launch_kernel(k, grid_for(n * 32, 32 * kWarps), 32 * kWarps, 0, st, pb, sp, n, list, fe, ge, he, state, flag,
                         (int)first);
}

cudaError_t lm_series_rows(const int* list, int64_t n, int T, int* rows, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    return launch_kernel(k_lm_series_rows, grid_for(n * T, 256), 256, 0, st, list, n, T, rows);
}

cudaError_t lm_series_output(const LmProblem& pb, const LmSeries& sp, int64_t n, double* state, double* x, double* cost,
                             double* grad, double* hess, double* cov, int32_t* info, cudaStream_t st) {
    auto k = pb.D <= 8 ? k_lm_series_output<8> : pb.D <= 16 ? k_lm_series_output<16> : k_lm_series_output<32>;
    if (n <= 0) return cudaSuccess;
    return launch_kernel(k, grid_for(n * 32, 32 * kWarps), 32 * kWarps, 0, st, pb, sp, n, state, x, cost, grad, hess, cov,
                         info);
}

}  // namespace gpe
