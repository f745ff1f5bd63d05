// Batched evaluation of the GP training objective and its gradient (SURVEY.md section 8f, rank 1).
//
// What it replaces: the inner loop of hyper-parameter fitting -- GaussianProcess.loglikelihood
// (gp_emulator/GaussianProcess.py:78-95) = _set_params -> _prepare_likelihood (:52-75: Z, Q = Z + noise I, inv(Q),
// invQ t, log|Q|) followed by partial_devs (:97-125) at the same theta.  The reference evaluates one theta at a time
// (5.5 ms at M = 250, D = 10 in numpy on the GPU box's 16 host cores); fitting a MultivariateEmulator runs n_pcs x n_tries independent L-BFGS-B
// descents on the SAME training inputs (multivariate_gp.py:176-186), so their evaluations batch: one CTA per
// (theta, target vector) problem, B problems per launch.
//
// Per problem (one 1024-thread CTA, matrices in an L2-resident workspace, vectors in shared memory):
//   1. Z_ij = b exp(-1/2 sum_d w_d (x_id - x_jd)^2), Q = Z + noise I                      (:61-69)
//   2. in-place block Gauss-Jordan inversion of Q without pivoting (Q is symmetric positive definite, so the
//      pivots are the LDL^T pivots: log|Q| = sum log p_k, and a pivot <= 0 is the reference's LinAlgError from
//      np.linalg.cholesky, :73-75).  NB pivots per pass (NB = 32 for M <= 256, 16 to 512, 8 beyond: what the staged
//      pivot rows / columns / coefficients leave room for in shared memory): M / NB rank-NB updates of the whole matrix on
//      the FP64 tensor cores (DMMA.8x8x4): M^3 FMA, 16 M^2 bytes of L2 traffic per NB pivots.  Round 1 ran NB = 8 and was
//      bound by the dependency chain of its M / 8 block steps, each streaming the matrix through L2 once
//      (profiles/r01_ncu_train_summary.md: DMMA pipe 15 %); NB = 32 makes 4x fewer, 4x heavier steps.
//   3. alpha = invQ t, t.alpha, alpha.alpha, trace(invQ)                                   (:71-72, :118-121)
//   4. g_d = -w_d/4 sum_ij (invQ_ij - alpha_i alpha_j) Z_ij (x_id - x_jd)^2,  g_D = 1/2 sum_ij (...) Z_ij,
//      g_{D+1} = noise/2 (trace(invQ) - alpha.alpha)                                       (:108-122)
//   loglik = 1/2 log|Q| + 1/2 t.alpha + M/2 log(2 pi)                                       (:90-92)
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <algorithm>
#include <mutex>
#include <vector>

#include "../../include/gpemu.h"
#include "gpe_math.cuh"
#include "host_common.h"
#include "launch.h"

namespace gpe {

constexpr int kTrainThreads = 512;    // 128 registers per thread: the rank-NB update keeps 8 accumulator tiles + 16 A fragments
constexpr int kTrainWarps = kTrainThreads / 32;

struct TrainParams {
    const double* x;        // (M, D) training inputs
    const double* targets;  // (T, M)
    const double* thetas;   // (B, D + 2)
    const int* tidx;        // (B) row of `targets` each problem fits
    double* work;           // (B, 2, Mp, Mp), Mp = M rounded up to 8: [0] Q -> invQ in place (identity in the padding), [1] Z
    double* loglik;         // (B)
    double* grad;           // (B, D + 2)
    int* status;            // (B) 0 ok, 1 Q not positive definite / non-finite
    int M, D;
    long long* trace;       // dev aid (normally null): CTA 0 adds its clock64() phase durations to trace[0..7]
};

// 1 / x for a positive, normal x without the division subroutine: hardware seed (>= 20 bits) + two Newton steps, ~60
// cycles of latency instead of ~400 -- it sits on the critical path of every pivot of the block inverse.
__device__ __forceinline__ double fast_rcp(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    e = fma(-x, r, 1.0);
    return fma(r, e, r);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Sum over the CTA, result in every thread (kTrainWarps <= 32: at most one partial per lane in the second stage).
__device__ __forceinline__ double block_sum(double v, double* red, int lane, int wid) {
    v = warp_sum(v);
    __syncthreads();  // `red` is free again
    if (lane == 0) red[wid] = v;
    __syncthreads();
    return warp_sum(lane < kTrainWarps ? red[lane] : 0.0);
}

// Work matrices are stored with pitch Mp = M rounded up to 8 and padded with the identity (Q_pad = diag(Q, I)), so
// that every 8 x 8 tile is full: inv(Q_pad) = diag(inv(Q), I), the padded pivots are 1 and add log 1 = 0.
// NB = pivots eliminated per pass over the matrix (8, 16 or 32; the last pass takes what is left, a multiple of 8).
template <int NB>
__global__ void __launch_bounds__(kTrainThreads, 1) k_train_eval(const TrainParams p) {
    constexpr int kNB = 8;            // DMMA tile edge
    constexpr int KK = NB / 4;        // DMMA k-steps of a full pass
    extern __shared__ __align__(16) double sm[];
    __shared__ double Pbuf[NB * NB];   // inverse of the pivot block
    __shared__ double rowbuf[2][NB];   // pivot row handed between the four warps of the block inverse
    __shared__ int s_bad;
    const int M = p.M, D = p.D, Mp = (M + 7) & ~7, nb = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int un = max(M * D, 3 * NB * Mp);
    double* xs = sm;                  // [M][D]                                    (phases 1 and 4)
    double* RrT = sm;                 // [KK][Mp][4]: RrT[kk][j][c] = A[k0 + 4 kk + c][j], the DMMA B operand (phase 2)
    double* Cc = sm + NB * Mp;        // [Mp][NB] pivot columns, staged
    double* CfT = sm + 2 * NB * Mp;   // [KK][Mp][4]: CfT[kk][i][c] = coef_i[4 kk + c], the DMMA A operand
    double* tt = sm + un;             // [M] targets
    double* alpha = tt + M;           // [M]
    double* ew = alpha + M;           // [D + 2] exp(theta)
    double* red = ew + 40;            // [32]
    double* A = p.work + (size_t)nb * 2 * Mp * Mp;
    double* Z = A + (size_t)Mp * Mp;

    const bool tracing = p.trace != nullptr && nb == 0 && tid == 0;
    long long tr_last = tracing ? clock64() : 0;
#define GPE_TR(k) do { if (tracing) { const long long now_ = clock64(); p.trace[k] += now_ - tr_last; tr_last = now_; } } while (0)
    for (int i = tid; i < M * D; i += kTrainThreads) xs[i] = p.x[i];
    const double* t = p.targets + (size_t)p.tidx[nb] * M;
    for (int i = tid; i < M; i += kTrainThreads) tt[i] = t[i];
    if (tid < D + 2) ew[tid] = exp(p.thetas[(size_t)nb * (D + 2) + tid]);
    if (tid == 0) s_bad = 0;
    __syncthreads();
    const double bb = ew[D], noise = ew[D + 1];

    // 1. covariance of the training set (reference GaussianProcess.py:61-69), identity in the padding
    for (int i = wid; i < Mp; i += kTrainWarps)
        for (int j = lane; j < Mp; j += 32) {
            if (i < M && j < M) {
                double r2 = 0.0;
                for (int d = 0; d < D; ++d) {
                    const double df = xs[i * D + d] - xs[j * D + d];
                    r2 += ew[d] * (df * df);
                }
                const double z = bb * exp_neg(-0.5 * r2);
                Z[i * Mp + j] = z;
                A[i * Mp + j] = (i == j) ? z + noise : z;
            } else {
                A[i * Mp + j] = (i == j) ? 1.0 : 0.0;
            }
        }
    __syncthreads();

    // 2. block Gauss-Jordan, NB pivots per pass.  With K the pivot index block, R = A[K, :], C = A[:, K], P = A[K, K]:
    //      A[K, K] <- inv(P),  A[K, J] <- inv(P) R,  A[I, K] <- -C inv(P),  A[I, J] <- A[I, J] - C inv(P) R
    //    i.e. every row i becomes  base_i + coef_i . R  with coef_i = inv(P)[i - k0, :] and base 0 for the pivot rows,
    //    coef_i = -C[i, :] inv(P) and base A[i, :] otherwise, except in the pivot columns where the new value is
    //    coef_i[j - k0].  That rank-NB update of the whole matrix runs on the FP64 tensor cores: per 8 x 8 tile NB / 4
    //    DMMA.8x8x4 with the accumulator fragment loaded from / stored to the L2-resident matrix ONCE per pass (16 bytes
    //    per lane, 64 contiguous bytes per row), operands pre-arranged in shared memory in fragment order
    //    (conflict-free); a warp owns two row tiles and half of the column tiles, so every B fragment it pulls from
    //    shared memory feeds two DMMAs.  inv(P) by scalar Gauss-Jordan inside the block (warp 0, entries in registers):
    //    its pivots are the LDL^T pivots of Q.
    double logdet = 0.0;
    bool bad = false;
    const int g = lane >> 2, c4 = lane & 3, ntile = Mp / kNB;
    GPE_TR(0);   // [0] inputs + covariance
    for (int k0 = 0; k0 < Mp; k0 += NB) {
        const int nbk = min(NB, Mp - k0);     // pivots of this pass (multiple of 8)
        const int kkn = nbk >> 2;             // its DMMA k-steps
        // pivot rows and columns, L2 -> shared memory (index arithmetic without integer division: Mp is a run-time value
        // and `e / Mp`, `e % Mp` per element made this the third most expensive step of the pass)
        for (int a = wid; a < nbk; a += kTrainWarps) {
            const double* src = A + (k0 + a) * Mp;
            double* dst = RrT + (a >> 2) * Mp * 4 + (a & 3);
#pragma unroll 4
            for (int j = lane; j < Mp; j += 32) dst[j * 4] = src[j];
        }
        __syncthreads();
        GPE_TR(1);   // [1] staging of the pivot rows
        // the pivot columns are staged by warps 4.. while warps 0-3 invert the pivot block (which only needs the rows)
        if (wid >= 4) {
            for (int e = tid - 128; e < Mp * NB; e += kTrainThreads - 128) {
                const int i = e / NB, a = e % NB;      // NB is a compile-time power of two
                if (a < nbk) Cc[e] = A[i * Mp + k0 + a];
            }
        } else {
            // inv(P) by scalar Gauss-Jordan in the registers of four warps (one per SM sub-partition): warp w owns rows
            // [w NB/4, (w + 1) NB/4) of the block, lane b column b.  Pivot step k: the owner of row k publishes it through a
            // double-buffered shared row + one 128-thread named barrier; column k restricted to a warp's rows sits in its lane
            // k (shuffles).  Per pivot the dependent chain is store -> barrier -> load -> reciprocal -> shuffle -> FMA, ~200
            // cycles; one warp holding the whole block (13 shuffles, 32 FMAs and the fix-ups per pivot) took 550, a CTA-wide
            // version with the block in shared memory 690.  The pivots are the LDL^T pivots of Q; their logarithms are
            // taken after the loop, one per lane of warp 0.  (A look-ahead variant -- one warp updates and inverts the NEXT
            // pivot block during the rank-NB update -- was measured and dropped: DFMA and DMMA share one FP64 pipe on this
            // GPU, so the inverse's dependent chain crawls behind the other warps' DMMAs: 366 k -> 545 k cycles in the
            // update for 99 k saved.)
            constexpr int RW = NB / 4;
            constexpr unsigned full = 0xffffffffu;
            double v[RW];
#pragma unroll
            for (int i = 0; i < RW; ++i) {
                const int ra = wid * RW + i, cb = lane;
                v[i] = (cb < NB) ? ((ra < nbk && cb < nbk) ? RrT[(ra >> 2) * Mp * 4 + (k0 + cb) * 4 + (ra & 3)] : ((ra == cb) ? 1.0 : 0.0)) : 0.0;
            }
            bool wbad = false;
            double mypiv = 1.0;
#pragma unroll
            for (int k = 0; k < NB; ++k) {
                if (k < nbk) {   // uniform over the four warps
                    const int ow = k / RW, ki = k % RW;
                    double* rb = rowbuf[k & 1];
                    if (wid == ow && lane < NB) rb[lane] = v[ki];
                    asm volatile("bar.sync 1, 128;" ::: "memory");
                    const double r = (lane < NB) ? rb[lane] : 0.0;     // P[k][my column]
                    const double piv = rb[k];
                    if (!(piv > 0.0) || !(piv < 1e300)) wbad = true;   // same value in all 128 threads
                    const double ip = fast_rcp(wbad ? 1.0 : piv);      // within an ulp or two of 1 / piv
#pragma unroll
                    for (int i = 0; i < RW; ++i) {
                        const double c = __shfl_sync(full, v[i], k & 31) * ip;   // P[my row i][k] / p
                        v[i] = (lane == k) ? -c : fma(-c, r, v[i]);
                    }
                    if (wid == ow) v[ki] = (lane == k) ? ip : r * ip;
                    if (wid == 0 && lane == (k & 31)) mypiv = piv;
                }
            }
#pragma unroll
            for (int i = 0; i < RW; ++i)
                if (lane < NB) Pbuf[(wid * RW + i) * NB + lane] = v[i];
            if (wid == 0) {
                if (wbad) { if (lane == 0) s_bad = 1; }
                else logdet += warp_sum(lane < nbk ? log(mypiv) : 0.0);
            }
        }
        __syncthreads();
        if (s_bad) { bad = true; break; }   // uniform
        const double* Ps = Pbuf;
        GPE_TR(2);   // [2] pivot-block inverse
        {   // coefficients: lane <-> column bq of inv(P) (kept in registers), 32 / NB rows per warp and sweep; the row of
            // pivot-column entries is read with 16-byte broadcast loads (the first version re-read inv(P) from shared
            // memory for every product and was bound by the shared-memory pipe)
            constexpr int RPW = 32 / NB;
            const int bq = lane % NB, sub = lane / NB;
            double pc[NB];
#pragma unroll
            for (int a = 0; a < NB; ++a) pc[a] = (a < nbk) ? Ps[a * NB + bq] : 0.0;
            for (int i = wid * RPW + sub; i < Mp; i += kTrainWarps * RPW) {
                const double2* crow = reinterpret_cast<const double2*>(Cc + i * NB);
                double s0 = 0.0, s1 = 0.0;
                if (nbk == NB) {               // full pass: no predicates, the broadcast loads are hoisted above the FMAs
#pragma unroll
                    for (int a2 = 0; a2 < NB / 2; ++a2) {
                        const double2 cv = crow[a2];
                        s0 = fma(cv.x, pc[2 * a2], s0);
                        s1 = fma(cv.y, pc[2 * a2 + 1], s1);
                    }
                } else {
#pragma unroll
                    for (int a2 = 0; a2 < NB / 2; ++a2) {
                        if (2 * a2 < nbk) {    // (nbk is a multiple of 8: whole pairs)
                            const double2 cv = crow[a2];
                            s0 = fma(cv.x, pc[2 * a2], s0);
                            s1 = fma(cv.y, pc[2 * a2 + 1], s1);
                        }
                    }
                }
                const bool prow = i >= k0 && i < k0 + nbk;
                if (bq < nbk) CfT[(bq >> 2) * Mp * 4 + i * 4 + (bq & 3)] = prow ? Ps[(i - k0) * NB + bq] : -(s0 + s1);
            }
        }
        __syncthreads();
        GPE_TR(3);   // [3] coefficients
        const int nct_half = (ntile + 1) >> 1, half = wid & 1;
        const int ct_begin = half * nct_half, ct_end = min(ntile, ct_begin + nct_half);
        for (int rp = wid >> 1; 2 * rp < ntile; rp += kTrainWarps / 2) {
            // two row tiles (the second may not exist: its rows are then never loaded or stored)
            const int i0a = 2 * rp * kNB, i0b = i0a + kNB;
            const bool has_b = 2 * rp + 1 < ntile;
            const bool prow_a = i0a >= k0 && i0a < k0 + nbk, prow_b = i0b >= k0 && i0b < k0 + nbk;
            double fa[KK], fb[KK];
#pragma unroll
            for (int kk = 0; kk < KK; ++kk) {
                fa[kk] = (kk < kkn) ? CfT[kk * Mp * 4 + (i0a + g) * 4 + c4] : 0.0;
                fb[kk] = (kk < kkn && has_b) ? CfT[kk * Mp * 4 + (i0b + g) * 4 + c4] : 0.0;
            }
            double* arow_a = A + (i0a + g) * Mp + 2 * c4;   // this lane's two accumulator columns of column tile 0
            double* arow_b = arow_a + kNB * Mp;
            for (int ct0 = ct_begin; ct0 < ct_end; ct0 += 4) {
                double2 ca[4], cb[4];
                if (kkn == KK && ct0 + 4 <= ct_end && has_b) {
                    // full batch of a full pass (every batch at M = 250): no predicates, so the eight B-fragment loads of a
                    // tile are hoisted above its sixteen DMMAs and the four tiles overlap
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        ca[q] = prow_a ? make_double2(0.0, 0.0) : *reinterpret_cast<const double2*>(arow_a + (ct0 + q) * kNB);
                        cb[q] = prow_b ? make_double2(0.0, 0.0) : *reinterpret_cast<const double2*>(arow_b + (ct0 + q) * kNB);
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int j0 = (ct0 + q) * kNB;
                        double bf[KK];
#pragma unroll
                        for (int kk = 0; kk < KK; ++kk) bf[kk] = RrT[kk * Mp * 4 + (j0 + g) * 4 + c4];
#pragma unroll
                        for (int kk = 0; kk < KK; ++kk) {
                            dmma_m8n8k4(ca[q].x, ca[q].y, fa[kk], bf[kk]);
                            dmma_m8n8k4(cb[q].x, cb[q].y, fb[kk], bf[kk]);
                        }
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int j0 = (ct0 + q) * kNB;
                        if (j0 >= k0 && j0 < k0 + nbk) {   // pivot columns: coef_i[j - k0], two consecutive entries per lane
                            const int bq = j0 - k0 + 2 * c4;
                            ca[q] = *reinterpret_cast<const double2*>(CfT + (bq >> 2) * Mp * 4 + (i0a + g) * 4 + (bq & 3));
                            cb[q] = *reinterpret_cast<const double2*>(CfT + (bq >> 2) * Mp * 4 + (i0b + g) * 4 + (bq & 3));
                        }
                        *reinterpret_cast<double2*>(arow_a + j0) = ca[q];
                        *reinterpret_cast<double2*>(arow_b + j0) = cb[q];
                    }
                    continue;
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    ca[q] = cb[q] = make_double2(0.0, 0.0);
                    if (ct0 + q < ct_end) {
                        if (!prow_a) ca[q] = *reinterpret_cast<const double2*>(arow_a + (ct0 + q) * kNB);
                        if (has_b && !prow_b) cb[q] = *reinterpret_cast<const double2*>(arow_b + (ct0 + q) * kNB);
                    }
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int j0 = (ct0 + q) * kNB;
                    if (ct0 + q < ct_end) {   // warp-uniform
#pragma unroll
                        for (int kk = 0; kk < KK; ++kk) {
                            if (kk < kkn) {
                                const double bf = RrT[kk * Mp * 4 + (j0 + g) * 4 + c4];
                                dmma_m8n8k4(ca[q].x, ca[q].y, fa[kk], bf);
                                dmma_m8n8k4(cb[q].x, cb[q].y, fb[kk], bf);
                            }
                        }
                        if (j0 >= k0 && j0 < k0 + nbk) {   // pivot columns: coef_i[j - k0], two consecutive entries per lane
                            const int bq = j0 - k0 + 2 * c4;
                            ca[q] = *reinterpret_cast<const double2*>(CfT + (bq >> 2) * Mp * 4 + (i0a + g) * 4 + (bq & 3));
                            if (has_b) cb[q] = *reinterpret_cast<const double2*>(CfT + (bq >> 2) * Mp * 4 + (i0b + g) * 4 + (bq & 3));
                        }
                        *reinterpret_cast<double2*>(arow_a + j0) = ca[q];
                        if (has_b) *reinterpret_cast<double2*>(arow_b + j0) = cb[q];
                    }
                }
            }
        }
        __syncthreads();
        GPE_TR(4);   // [4] rank-NB update
    }
    const int G = D + 2;
    if (bad) {
        if (tid == 0) {
            p.status[nb] = 1;
            p.loglik[nb] = nan("");
            for (int d = 0; d < G; ++d) p.grad[(size_t)nb * G + d] = nan("");
        }
        return;
    }
    for (int i = tid; i < M * D; i += kTrainThreads) xs[i] = p.x[i];   // the staging buffers overwrote the inputs
    __syncthreads();

    // 3. alpha = invQ t and the scalar sums
    for (int i = wid; i < M; i += kTrainWarps) {
        const double* ai = A + i * Mp;
        double s = 0.0;
        for (int j0 = lane; j0 < M; j0 += 256) {
            double v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = (j0 + 32 * u < M) ? ai[j0 + 32 * u] : 0.0;
#pragma unroll
            for (int u = 0; u < 8; ++u)
                if (j0 + 32 * u < M) s = fma(v[u], tt[j0 + 32 * u], s);
        }
        s = warp_sum(s);
        if (lane == 0) alpha[i] = s;
    }
    __syncthreads();
    double s_ta = 0.0, s_aa = 0.0, s_tr = 0.0;
    for (int i = tid; i < M; i += kTrainThreads) {
        s_ta = fma(tt[i], alpha[i], s_ta);
        s_aa = fma(alpha[i], alpha[i], s_aa);
        s_tr += A[i * Mp + i];
    }
    s_ta = block_sum(s_ta, red, lane, wid);
    s_aa = block_sum(s_aa, red, lane, wid);
    s_tr = block_sum(s_tr, red, lane, wid);
    GPE_TR(5);   // [5] alpha and scalar sums

    // 4. gradient sums  S_d = sum_ij (invQ_ij - alpha_i alpha_j) Z_ij (x_id - x_jd)^2  (d < D)  and  S_D = sum_ij (...) Z_ij,
    //    kGS accumulators per pass over the two matrices, four rows in flight per thread
    constexpr int kGS = 12;   // D = 10: all eleven sums in ONE pass over the two matrices (the 64-register version took two)
    for (int d0 = 0; d0 <= D; d0 += kGS) {
        double acc[kGS];
#pragma unroll
        for (int dd = 0; dd < kGS; ++dd) acc[dd] = 0.0;
        for (int j = lane; j < M; j += 32) {
            const double aj = alpha[j];
            double xj[kGS];
#pragma unroll
            for (int dd = 0; dd < kGS; ++dd) xj[dd] = (d0 + dd < D) ? xs[j * D + d0 + dd] : 0.0;
            for (int i0 = wid; i0 < M; i0 += 4 * kTrainWarps) {
                double va[4], vz[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int i = i0 + q * kTrainWarps;
                    va[q] = (i < M) ? A[i * Mp + j] : 0.0;
                    vz[q] = (i < M) ? Z[i * Mp + j] : 0.0;
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int i = i0 + q * kTrainWarps;
                    if (i < M) {
                        const double wz = fma(-alpha[i], aj, va[q]) * vz[q];
#pragma unroll
                        for (int dd = 0; dd < kGS; ++dd) {
                            const int d = d0 + dd;
                            if (d < D) {
                                const double df = xs[i * D + d] - xj[dd];
                                acc[dd] = fma(wz * df, df, acc[dd]);
                            } else if (d == D) {
                                acc[dd] += wz;
                            }
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int dd = 0; dd < kGS; ++dd) {
            const int d = d0 + dd;
            if (d <= D) {   // uniform
                const double sum = block_sum(acc[dd], red, lane, wid);
                if (tid == 0) p.grad[(size_t)nb * G + d] = (d < D) ? -0.25 * ew[d] * sum : 0.5 * sum;
            }
        }
    }
    GPE_TR(6);   // [6] gradient sums
#undef GPE_TR
    if (tid == 0) {
        p.grad[(size_t)nb * G + D + 1] = 0.5 * noise * (s_tr - s_aa);
        const double ll = 0.5 * logdet + 0.5 * s_ta + 0.5 * (double)M * 1.8378770664093453;  // log(2 pi)
        p.loglik[nb] = ll;
        // positive pivots but an overflowed / NaN result (e.g. a numerically singular Q): report it like a failed
        // factorisation rather than handing non-finite numbers to the optimiser
        bool finite = isfinite(ll);
        for (int d = 0; d < G; ++d) finite = finite && isfinite(p.grad[(size_t)nb * G + d]);
        p.status[nb] = finite ? 0 : 1;
        if (!finite) {
            p.loglik[nb] = nan("");
            for (int d = 0; d < G; ++d) p.grad[(size_t)nb * G + d] = nan("");
        }
    }
}

}  // namespace gpe

using namespace gpe;

struct gpe_trainer {
    int device = 0, M = 0, D = 0, T = 0, sms = 0;
    int NB = 8;                   // pivots per pass of the block Gauss-Jordan (k_train_eval<NB>)
    cudaStream_t st = nullptr;
    double* d_x = nullptr;
    double* d_targets = nullptr;
    double* d_work = nullptr;     // capacity `cap` problems
    double* d_theta = nullptr;    // cap x (D + 2)
    double* d_ll = nullptr;
    double* d_grad = nullptr;
    int* d_tidx = nullptr;
    int* d_status = nullptr;
    int cap = 0;
    size_t smem = 0;
    std::mutex mu;                // evaluations on one trainer share its workspace
};

namespace {

long long* g_train_trace = nullptr;   // dev aid: gpe_debug_train_trace

#define TR_TRY(expr)                                                                                              \
    do {                                                                                                          \
        cudaError_t _e = (expr);                                                                                  \
        if (_e != cudaSuccess)                                                                                    \
            return set_error(GPE_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

void free_batch_buffers(gpe_trainer* t) {
    if (t->d_work) cudaFree(t->d_work);
    if (t->d_theta) cudaFree(t->d_theta);
    if (t->d_ll) cudaFree(t->d_ll);
    if (t->d_grad) cudaFree(t->d_grad);
    if (t->d_tidx) cudaFree(t->d_tidx);
    if (t->d_status) cudaFree(t->d_status);
    t->d_work = t->d_theta = t->d_ll = t->d_grad = nullptr;
    t->d_tidx = t->d_status = nullptr;
    t->cap = 0;
}

int reserve(gpe_trainer* t, int nb) {
    if (nb <= t->cap) return GPE_OK;
    free_batch_buffers(t);
    const size_t G = (size_t)t->D + 2, mp = ((size_t)t->M + 7) / 8 * 8, mm = mp * mp;
    TR_TRY(cudaMalloc((void**)&t->d_work, (size_t)nb * 2 * mm * 8));
    TR_TRY(cudaMalloc((void**)&t->d_theta, (size_t)nb * G * 8));
    TR_TRY(cudaMalloc((void**)&t->d_ll, (size_t)nb * 8));
    TR_TRY(cudaMalloc((void**)&t->d_grad, (size_t)nb * G * 8));
    TR_TRY(cudaMalloc((void**)&t->d_tidx, (size_t)nb * sizeof(int)));
    TR_TRY(cudaMalloc((void**)&t->d_status, (size_t)nb * sizeof(int)));
    t->cap = nb;
    return GPE_OK;
}

}  // namespace

extern "C" {

// Developer aid (not part of the public header): CTA 0 of k_train_eval adds the clock64() duration of each phase to
// device_buf[0..7] (inputs + covariance, staging, pivot inverse, coefficients, update, alpha, gradient sums); NULL = off.
void gpe_debug_train_trace(long long* device_buf) { g_train_trace = device_buf; }

int gpe_trainer_create(int device, int M, int D, int T, const double* inputs, const double* targets, gpe_trainer** out) {
    if (!out) return set_error(GPE_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (M < 1 || D < 1 || T < 1) return set_error(GPE_ERR_INVALID, "need M >= 1, D >= 1, T >= 1 (got %d, %d, %d)", M, D, T);
    if (D > GPE_TRAIN_MAX_D) return set_error(GPE_ERR_UNSUPPORTED, "D = %d exceeds GPE_TRAIN_MAX_D = %d", D, GPE_TRAIN_MAX_D);
    if (M > GPE_TRAIN_MAX_M) return set_error(GPE_ERR_UNSUPPORTED, "M = %d exceeds GPE_TRAIN_MAX_M = %d", M, GPE_TRAIN_MAX_M);
    if (!inputs || !targets) return set_error(GPE_ERR_INVALID, "inputs / targets is NULL");
    // pivots per pass: the largest of 32, 16, 8 whose staged pivot rows, columns and coefficients (3 NB Mp doubles) fit
    // beside the vectors and the kernel's static shared memory (pivot block NB^2 doubles)
    const size_t mp8 = ((size_t)M + 7) / 8 * 8;
    int NB = 32;
    size_t smem = 0;
    for (;; NB /= 2) {
        smem = (std::max((size_t)M * D, (size_t)3 * NB * mp8) + 2 * (size_t)M + 40 + 32) * 8;
        if (smem + (size_t)NB * NB * 8 + 1024 <= 232448 || NB == 8) break;
    }
    if (smem + (size_t)NB * NB * 8 + 1024 > 232448)
        return set_error(GPE_ERR_UNSUPPORTED, "M x D = %d x %d needs %zu bytes of shared memory per CTA", M, D, smem);
    int sms = 0;
    int rc = require_device(device, &sms);
    if (rc) return rc;
    TR_TRY(cudaSetDevice(device));
    gpe_trainer* t = new gpe_trainer;
    t->device = device; t->M = M; t->D = D; t->T = T; t->sms = sms; t->smem = smem; t->NB = NB;
    cudaError_t e = cudaStreamCreateWithFlags(&t->st, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc((void**)&t->d_x, (size_t)M * D * 8);
    if (e == cudaSuccess) e = cudaMalloc((void**)&t->d_targets, (size_t)T * M * 8);
    if (e == cudaSuccess) e = cudaMemcpy(t->d_x, inputs, (size_t)M * D * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(t->d_targets, targets, (size_t)T * M * 8, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        gpe_trainer_destroy(t);
        return set_error(GPE_ERR_CUDA, "trainer setup failed: %s", cudaGetErrorString(e));
    }
    *out = t;
    return GPE_OK;
}

int gpe_trainer_destroy(gpe_trainer* t) {
    if (!t) return GPE_OK;
    cudaSetDevice(t->device);
    free_batch_buffers(t);
    if (t->d_x) cudaFree(t->d_x);
    if (t->d_targets) cudaFree(t->d_targets);
    if (t->st) cudaStreamDestroy(t->st);
    delete t;
    return GPE_OK;
}

int gpe_trainer_eval(gpe_trainer* t, int B, const int* target_index, const double* thetas, double* loglik, double* grad,
                     int* status) {
    NvtxRange nvtx_range("gpe_trainer_eval");
    if (!t) return set_error(GPE_ERR_INVALID, "trainer is NULL");
    if (B < 0) return set_error(GPE_ERR_INVALID, "B must be >= 0");
    if (B == 0) return GPE_OK;
    if (!thetas || !loglik || !grad || !status) return set_error(GPE_ERR_INVALID, "thetas / loglik / grad / status is NULL");
    if (target_index)
        for (int i = 0; i < B; ++i)
            if (target_index[i] < 0 || target_index[i] >= t->T)
                return set_error(GPE_ERR_INVALID, "target_index[%d] = %d out of range [0, %d)", i, target_index[i], t->T);
    std::lock_guard<std::mutex> lock(t->mu);
    TR_TRY(cudaSetDevice(t->device));
    const size_t G = (size_t)t->D + 2, mp = ((size_t)t->M + 7) / 8 * 8, mm = mp * mp;
    // problems per launch: whole waves of CTAs, workspace bounded by 4 GB
    const int by_mem = (int)std::max<size_t>(1, ((size_t)4 << 30) / (2 * mm * 8));
    const int chunk = std::min(B, std::min(by_mem, 8 * t->sms));
    int rc = reserve(t, chunk);
    if (rc) return rc;
    std::vector<int> zeros;
    if (!target_index) zeros.assign((size_t)chunk, 0);
    for (int b0 = 0; b0 < B; b0 += chunk) {
        const int nb = std::min(chunk, B - b0);
        TR_TRY(cudaMemcpyAsync(t->d_theta, thetas + (size_t)b0 * G, (size_t)nb * G * 8, cudaMemcpyHostToDevice, t->st));
        TR_TRY(cudaMemcpyAsync(t->d_tidx, target_index ? target_index + b0 : zeros.data(), (size_t)nb * sizeof(int),
                               cudaMemcpyHostToDevice, t->st));
        TrainParams p;
        p.x = t->d_x; p.targets = t->d_targets; p.thetas = t->d_theta; p.tidx = t->d_tidx; p.work = t->d_work;
        p.loglik = t->d_ll; p.grad = t->d_grad; p.status = t->d_status; p.M = t->M; p.D = t->D;
        p.trace = g_train_trace;
        auto kern = t->NB == 32 ? k_train_eval<32> : (t->NB == 16 ? k_train_eval<16> : k_train_eval<8>);
        TR_TRY(launch_kernel(kern, nb, kTrainThreads, t->smem, t->st, p));
        TR_TRY(cudaMemcpyAsync(loglik + b0, t->d_ll, (size_t)nb * 8, cudaMemcpyDeviceToHost, t->st));
        TR_TRY(cudaMemcpyAsync(grad + (size_t)b0 * G, t->d_grad, (size_t)nb * G * 8, cudaMemcpyDeviceToHost, t->st));
        TR_TRY(cudaMemcpyAsync(status + b0, t->d_status, (size_t)nb * sizeof(int), cudaMemcpyDeviceToHost, t->st));
        TR_TRY(cudaStreamSynchronize(t->st));
    }
    return GPE_OK;
}

}  // extern "C"
