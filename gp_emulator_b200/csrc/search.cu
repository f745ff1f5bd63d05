// Candidate search (DESIGN 4.6e): per pixel, the k candidates of a table with the smallest misfit, ranked without
// forming a residual per wavelength.  With m_k the bank means at candidate k (E values),
//   cost_nk = a_k + s_n . m_k + c_n
//     band cost:      a_k = 1/2 sum_e w_e m_ke^2     s_n = -w o o_n
//     spectrum cost:  a_k = 1/2 m_k^T C m_k          s_n = -basis . (l o o_n)     C = basis . diag(l) . basis^T
// and c_n is constant within a pixel, so the ranking score a_k + s_n . m_k is a skinny FP64 GEMM (N x E) . (E x K) plus a
// column constant, followed by a top-k per row.  The (N, K) score matrix never leaves the SM: k_search_topk keeps, per
// thread and row, a sorted list of its best (score, index) pairs in registers.  The exact costs of the winners are formed
// afterwards by the per-wavelength cost kernels (gpemu.cu): the expanded form only chooses, it is never returned.
//
// Order: (score, candidate index), lexicographic.  A NaN score compares false and is never inserted; an empty slot is
// (+inf, kSrEmpty), which any selectable candidate (+inf included) beats.  Every score is computed by the same sequence
// of DMMA k-steps whatever CTA or position it lands in, so the selected set depends on neither the split of the
// candidates over CTAs nor on the pixels a launch holds.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <algorithm>

#include "gpe_math.cuh"
#include "gpe_ptx.cuh"
#include "launch.h"

namespace gpe {

constexpr int kSrThreads = 256, kSrRows = 128, kSrCols = 128;   // CTA: 8 warps x 16 pixel rows; candidate groups of 128
constexpr int kSrEmpty = 0x7fffffff;

__device__ __forceinline__ bool sr_better(double v, int i, double w, int j) { return v < w || (v == w && i < j); }

// Insert (v, i) into the ascending list; the caller has checked that it beats the last entry.
template <int KM>
__device__ __forceinline__ void sr_insert(double (&lv)[KM], int (&li)[KM], double v, int i) {
#pragma unroll
    for (int j = KM - 1; j > 0; --j) {
        const bool up = sr_better(v, i, lv[j - 1], li[j - 1]);   // the new entry lands above j - 1: slot j takes j - 1
        const bool here = !up && sr_better(v, i, lv[j], li[j]);
        lv[j] = up ? lv[j - 1] : (here ? v : lv[j]);
        li[j] = up ? li[j - 1] : (here ? i : li[j]);
    }
    if (sr_better(v, i, lv[0], li[0])) { lv[0] = v; li[0] = i; }
}

// Merge the list with the one of lane ^ mask, keeping the best KM (KM a power of two): the element-wise better of the
// list and the partner's reversed list is bitonic and holds the best KM of both; a bitonic half-cleaner cascade sorts
// it.  Both lanes end with the same list.
template <int KM>
__device__ __forceinline__ void sr_merge_lanes(double (&lv)[KM], int (&li)[KM], int mask) {
    // slots j and KM - 1 - j together: both partner values are read before either slot changes (no copy of the list)
#pragma unroll
    for (int j = 0; j < (KM + 1) / 2; ++j) {
        const int q = KM - 1 - j;
        const double pq = __shfl_xor_sync(0xffffffffu, lv[q], mask), pj = __shfl_xor_sync(0xffffffffu, lv[j], mask);
        const int iq = __shfl_xor_sync(0xffffffffu, li[q], mask), ij = __shfl_xor_sync(0xffffffffu, li[j], mask);
        if (sr_better(pq, iq, lv[j], li[j])) { lv[j] = pq; li[j] = iq; }
        if (q != j && sr_better(pj, ij, lv[q], li[q])) { lv[q] = pj; li[q] = ij; }
    }
#pragma unroll
    for (int s = KM / 2; s > 0; s >>= 1)
#pragma unroll
        for (int j = 0; j < KM; ++j)
            if ((j & s) == 0 && sr_better(lv[j + s], li[j + s], lv[j], li[j])) {
                const double tv = lv[j]; const int ti = li[j];
                lv[j] = lv[j + s]; li[j] = li[j + s];
                lv[j + s] = tv; li[j + s] = ti;
            }
}

// Top-KM of every pixel row against the candidate table.
//   s (R, E): pixel operands; tbl [KS][Kp][4]: candidate means, k-block contiguous like the basis image (zero past E);
//   ta (Kp): a_k, NaN past K.  Warp w owns rows 16 w .. 16 w + 15 of the CTA tile and keeps their s as A fragments in
//   registers; candidate groups g = blockIdx.y, blockIdx.y + gridDim.y, ... arrive by TMA bulk copies through a two-stage
//   mbarrier ring; a_k is the accumulators' initial value.  Lane (row r, columns 2 (lane % 4) + h) compares each score with
//   its list's last entry and inserts the winners; at the end the four lanes of a row merge their lists.
//   gridDim.y == 1: the first k indices of each row go to sel (R, k) (-1: empty).  Otherwise the CTA's list goes to
//   part_v / part_i [gridDim.y][R][k] for k_search_merge.
template <int KS, int KM>
__global__ void __launch_bounds__(kSrThreads, 1) k_search_topk(const double* __restrict__ s, int64_t R, int E,
                                                                const double* __restrict__ tbl, const double* __restrict__ ta,
                                                                int Kp, int k, int64_t* __restrict__ sel,
                                                                double* __restrict__ part_v, int* __restrict__ part_i) {
    extern __shared__ __align__(128) unsigned char ssm[];
    constexpr uint32_t stage_doubles = (uint32_t)KS * kSrCols * 4 + kSrCols, ks_bytes = kSrCols * 4 * 8;
    uint64_t* full = reinterpret_cast<uint64_t*>(ssm);          // [2]
    double* stage = reinterpret_cast<double*>(ssm + 128);       // [2][KS][128][4] + [2][128] a_k
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    smem_guard(128u + 2u * stage_doubles * 8u);
    const int64_t t0 = (int64_t)blockIdx.x * kSrRows;
    const int gy = (int)gridDim.y, y0 = (int)blockIdx.y, ngroups = Kp / kSrCols;
    const int ng = (ngroups - y0 + gy - 1) / gy;
    if (tid == 0) {
        mbar_init(&full[0], 1);
        mbar_init(&full[1], 1);
        fence_mbar_init();
    }
    __syncthreads();
    auto load_group = [&](int it, int st) {   // thread 0
        const int g = y0 + it * gy;
        double* dst = stage + (size_t)st * stage_doubles;
        mbar_arrive_expect_tx(&full[st], (uint32_t)KS * ks_bytes + kSrCols * 8);
        for (int ks = 0; ks < KS; ++ks)
            tma_bulk_g2s(dst + (size_t)ks * kSrCols * 4, tbl + ((size_t)ks * Kp + (size_t)g * kSrCols) * 4, ks_bytes, &full[st]);
        tma_bulk_g2s(dst + (size_t)KS * kSrCols * 4, ta + (size_t)g * kSrCols, kSrCols * 8, &full[st]);
    };
    if (tid == 0) {
        if (ng > 0) load_group(0, 0);
        if (ng > 1) load_group(1, 1);
    }
    // A fragments: lane holds s[row = 16 warp + 8 i + lane / 4][e = 4 ks + lane % 4]
    double a[2][KS];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const int64_t r = t0 + 16 * warp + 8 * i + (lane >> 2);
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
            const int e = 4 * ks + (lane & 3);
            a[i][ks] = (r < R && e < E) ? s[r * E + e] : 0.0;
        }
    }
    double lv[2][KM];
    int li[2][KM];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < KM; ++j) { lv[i][j] = __longlong_as_double(0x7ff0000000000000LL); li[i][j] = kSrEmpty; }
    // candidates per sub-block: NJ n-tiles of 8 (fewer accumulators where the A fragments and the lists fill the registers)
    constexpr int NJ = KS * KM >= 384 ? (KS >= 24 ? 1 : 2) : 4;
    uint32_t par = 0;
    for (int it = 0; it < ng; ++it) {
        const int st = it & 1;
        mbar_wait(&full[st], (par >> st) & 1u);
        par ^= 1u << st;
        const double* sb = stage + (size_t)st * stage_doubles;
        const int cbase = (y0 + it * gy) * kSrCols;
#pragma unroll 1
        for (int sub = 0; sub < kSrCols; sub += 8 * NJ) {
            double acc[2][NJ][2];
#pragma unroll
            for (int j = 0; j < NJ; ++j)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const double a0 = sb[KS * kSrCols * 4 + sub + 8 * j + 2 * (lane & 3) + h];
                    acc[0][j][h] = a0;
                    acc[1][j][h] = a0;
                }
            const double* bs = sb + (size_t)(sub + (lane >> 2)) * 4 + (lane & 3);
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    // B[k = lane % 4][n = lane / 4] = m[candidate sub + 8 j + lane / 4][e = 4 ks + lane % 4]
                    const double bf = bs[(size_t)ks * kSrCols * 4 + j * 32];
#pragma unroll
                    for (int i = 0; i < 2; ++i) dmma_m8n8k4(acc[i][j][0], acc[i][j][1], a[i][ks], bf);
                }
            }
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < NJ; ++j)
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int c = cbase + sub + 8 * j + 2 * (lane & 3) + h;
                        if (sr_better(acc[i][j][h], c, lv[i][KM - 1], li[i][KM - 1])) sr_insert<KM>(lv[i], li[i], acc[i][j][h], c);
                    }
        }
        __syncthreads();   // every warp is done with this stage: refill it
        if (tid == 0 && it + 2 < ng) load_group(it + 2, st);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        sr_merge_lanes<KM>(lv[i], li[i], 1);
        sr_merge_lanes<KM>(lv[i], li[i], 2);
    }
    if ((lane & 3) != 0) return;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const int64_t r = t0 + 16 * warp + 8 * i + (lane >> 2);
        if (r >= R) continue;
#pragma unroll
        for (int j = 0; j < KM; ++j) {
            if (j >= k) break;
            if (gy == 1) {
                sel[r * k + j] = li[i][j] == kSrEmpty ? -1 : (int64_t)li[i][j];
            } else {
                part_v[((size_t)y0 * R + r) * k + j] = lv[i][j];
                part_i[((size_t)y0 * R + r) * k + j] = li[i][j];
            }
        }
    }
}

// Candidate-split calls: the best k of the gy partial lists of every row, in (score, index) order.
template <int KM>
__global__ void k_search_merge(const double* __restrict__ part_v, const int* __restrict__ part_i, int64_t R, int k, int gy,
                               int64_t* __restrict__ sel) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (int64_t)gridDim.x * blockDim.x) {
        double lv[KM];
        int li[KM];
#pragma unroll
        for (int j = 0; j < KM; ++j) { lv[j] = __longlong_as_double(0x7ff0000000000000LL); li[j] = kSrEmpty; }
        for (int y = 0; y < gy; ++y)
            for (int j = 0; j < k; ++j) {
                const double v = part_v[((size_t)y * R + r) * k + j];
                const int i = part_i[((size_t)y * R + r) * k + j];
                if (i != kSrEmpty && sr_better(v, i, lv[KM - 1], li[KM - 1])) sr_insert<KM>(lv, li, v, i);
            }
#pragma unroll
        for (int j = 0; j < KM; ++j)
            if (j < k) sel[r * k + j] = li[j] == kSrEmpty ? -1 : (int64_t)li[j];
    }
}

// Candidate table: tbl [ksa][Kp][4] = the means mu (K, E), zero past E and K; ta (Kp) = a_k, NaN past K.
//   band cost (C == NULL):  a_k = 1/2 sum_e w_e m_ke^2        (w == NULL: 1)
//   spectrum cost:          a_k = 1/2 sum_e m_ke (sum_f C_ef m_kf)
__global__ void k_search_table(const double* __restrict__ mu, int64_t K, int E, int ksa, int Kp, const double* __restrict__ w,
                               const double* __restrict__ C, double* __restrict__ tbl, double* __restrict__ ta) {
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < Kp; c += (int64_t)gridDim.x * blockDim.x) {
        const double* m = mu + c * E;
        for (int e = 0; e < 4 * ksa; ++e) tbl[((size_t)(e >> 2) * Kp + c) * 4 + (e & 3)] = (c < K && e < E) ? m[e] : 0.0;
        if (c >= K) {
            ta[c] = __longlong_as_double(0x7ff8000000000000LL);
            continue;
        }
        double v = 0.0;
        if (C) {
            for (int e = 0; e < E; ++e) {
                double t = 0.0;
                for (int f = 0; f < E; ++f) t = fma(C[(size_t)e * E + f], m[f], t);
                v = fma(m[e], t, v);
            }
        } else {
            for (int e = 0; e < E; ++e) v = fma((w ? w[e] : 1.0) * m[e], m[e], v);
        }
        ta[c] = 0.5 * v;
    }
}

// Band-cost pixel operand: s (R, E) = -(w o obs_r).
__global__ void k_search_band_s(const double* __restrict__ obs, int64_t obs_ld, const double* __restrict__ w, int64_t R, int E,
                                double* __restrict__ s) {
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < R * E; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = q / E;
        const int e = (int)(q - r * E);
        s[q] = -((w ? w[e] : 1.0) * obs[r * obs_ld + e]);
    }
}

// Per-point weights (DESIGN 4.6f): both costs stay a_k + s_n . m'_k + c_n with a wider pixel operand and table row, and
// a_k = 0 (NaN past K):
//   band cost:      m'_k = [1/2 m_k o m_k, m_k] (2E)                pixel [w_n, -w_n o o_n]
//   spectrum cost:  m'_k = [m_ke m_kf for e <= f, m_k] (E(E+1)/2 + E)   pixel [C_n upper triangle, diagonal halved, s_n]
// (the upper triangle row by row).  tbl [search_ks(Ew)][Kp][4], zero past Ew and K.
__global__ void k_search_table_pw(const double* __restrict__ mu, int64_t K, int E, int Ew, int ksa, int Kp, bool spectra,
                                  double* __restrict__ tbl, double* __restrict__ ta) {
    const int nq = spectra ? E * (E + 1) / 2 : E;
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < Kp; c += (int64_t)gridDim.x * blockDim.x) {
        const double* m = mu + c * E;
        int e = 0, f = 0;
        for (int q = 0; q < 4 * ksa; ++q) {
            double v = 0.0;
            if (c < K && q < nq) {
                v = spectra ? m[e] * m[f] : 0.5 * (m[q] * m[q]);
                if (spectra && ++f == E) { ++e; f = e; }
            } else if (c < K && q < Ew) {
                v = m[q - nq];
            }
            tbl[((size_t)(q >> 2) * Kp + c) * 4 + (q & 3)] = v;
        }
        ta[c] = c < K ? 0.0 : __longlong_as_double(0x7ff8000000000000LL);
    }
}

// Per-point-weight pixel operand op (R, Ew): band [w_r, -(w_r o obs_r)]; spectrum [C_r (e <= f, diagonal halved), s_r] from
// the curvature Cn (R, E, E) and s (R, E).
__global__ void k_search_operand_pw(const double* __restrict__ obs, int64_t obs_ld, const double* __restrict__ w, int64_t w_ld,
                                    const double* __restrict__ s, const double* __restrict__ Cn, int64_t R, int E, int Ew,
                                    bool spectra, double* __restrict__ op) {
    const int nq = spectra ? E * (E + 1) / 2 : E;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < R * Ew; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = q / Ew;
        const int j = (int)(q - r * Ew);
        double v;
        if (!spectra) {
            v = j < E ? w[r * w_ld + j] : -(w[r * w_ld + j - E] * obs[r * obs_ld + j - E]);
        } else if (j < nq) {
            int e = 0, t = j;
            while (t >= E - e) { t -= E - e; ++e; }
            const int f = e + t;
            v = Cn[(r * E + e) * E + f];
            if (e == f) v *= 0.5;
        } else {
            v = s[r * E + j - nq];
        }
        op[q] = v;
    }
}

// x (R, D) = cand[sel[r, j]] (candidate 0 for an empty slot: its cost is discarded).
__global__ void k_search_gather(const double* __restrict__ cand, int D, const int64_t* __restrict__ sel, int k, int j, int64_t R,
                                double* __restrict__ x) {
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < R * D; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = q / D;
        const int d = (int)(q - r * D);
        const int64_t c = sel[r * k + j];
        x[q] = cand[(c < 0 ? 0 : c) * D + d];
    }
}

// Final order of each row: ascending (exact cost, index), NaN costs after every number, empty slots (idx -1, cost NaN)
// last.  cst [k][R] holds the exact cost of slot j of row r; one thread per (row, slot) writes the entry at its rank.
__device__ __forceinline__ bool sr_before(double c1, int64_t i1, double c2, int64_t i2) {
    if (i1 < 0) return false;
    if (i2 < 0) return true;
    const bool n1 = isnan(c1), n2 = isnan(c2);
    if (n1 != n2) return n2;
    if (!n1 && c1 != c2) return c1 < c2;
    return i1 < i2;
}

__global__ void k_search_output(const int64_t* __restrict__ sel, const double* __restrict__ cst, int64_t R, int k,
                                int64_t* __restrict__ idx, double* __restrict__ cost) {
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < R * k; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = q / k;
        const int j = (int)(q - r * k);
        const int64_t ij = sel[q];
        const double cj = cst[(size_t)j * R + r];
        int rank = 0;
        for (int j2 = 0; j2 < k; ++j2)
            if (j2 != j && sr_before(cst[(size_t)j2 * R + r], sel[r * k + j2], cj, ij)) ++rank;
        if (ij < 0) {   // empty slots are all equal: keep their slot order
            rank = 0;
            for (int j2 = 0; j2 < k; ++j2) rank += sel[r * k + j2] >= 0 || j2 < j;
        }
        if (idx) idx[r * k + rank] = ij;
        if (cost) cost[r * k + rank] = ij < 0 ? __longlong_as_double(0x7ff8000000000000LL) : cj;
    }
}

namespace {
inline unsigned grid_for(int64_t n, int threads) { return (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + threads - 1) / threads, 4096)); }
inline int km_for(int k) { return k <= 1 ? 1 : k <= 2 ? 2 : k <= 4 ? 4 : k <= 8 ? 8 : 16; }
}  // namespace

int search_ks(int E) {
    const int ks = (E + 3) / 4;
    return ks <= 3 ? 3 : ks <= 5 ? 5 : ks <= 8 ? 8 : ks <= 12 ? 12 : ks <= 16 ? 16 : 24;
}

size_t search_smem(int E) { return 128 + 2 * ((size_t)search_ks(E) * kSrCols * 4 + kSrCols) * 8; }

int search_pad(int64_t K) { return (int)((K + kSrCols - 1) / kSrCols * kSrCols); }

int search_split(int64_t call_N, int64_t K) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int64_t tiles = (call_N + kSrRows - 1) / kSrRows, ngroups = (K + kSrCols - 1) / kSrCols;
    return (int)std::max<int64_t>(1, std::min<int64_t>(ngroups, (int64_t)sms / std::max<int64_t>(tiles, 1)));
}

cudaError_t search_table(const double* mu, int64_t K, int E, int Kp, const double* w, const double* C, double* tbl, double* ta,
                         cudaStream_t st) {
    return launch_kernel(k_search_table, grid_for(Kp, 128), 128, 0, st, mu, K, E, search_ks(E), Kp, w, C, tbl, ta);
}

cudaError_t search_table_pw(const double* mu, int64_t K, int E, int Ew, int Kp, bool spectra, double* tbl, double* ta, cudaStream_t st) {
    return launch_kernel(k_search_table_pw, grid_for(Kp, 128), 128, 0, st, mu, K, E, Ew, search_ks(Ew), Kp, spectra, tbl, ta);
}

cudaError_t search_operand_pw(const double* obs, int64_t obs_ld, const double* w, int64_t w_ld, const double* s, const double* Cn,
                              int64_t R, int E, int Ew, bool spectra, double* op, cudaStream_t st) {
    return launch_kernel(k_search_operand_pw, grid_for(R * Ew, 256), 256, 0, st, obs, obs_ld, w, w_ld, s, Cn, R, E, Ew, spectra, op);
}

cudaError_t search_band_s(const double* obs, int64_t obs_ld, const double* w, int64_t R, int E, double* s, cudaStream_t st) {
    return launch_kernel(k_search_band_s, grid_for(R * E, 256), 256, 0, st, obs, obs_ld, w, R, E, s);
}

cudaError_t search_topk(const double* s, int64_t R, int E, const double* tbl, const double* ta, int Kp, int k, int gy,
                        double* part_v, int* part_i, int64_t* sel, cudaStream_t st) {
    const int ks = search_ks(E), km = km_for(k);
    const dim3 grid((unsigned)((R + kSrRows - 1) / kSrRows), (unsigned)gy);
    const size_t smem = search_smem(E);
    cudaError_t e = cudaErrorInvalidValue;
#define GPE_SR_KM(KSV)                                                                                                      \
    switch (km) {                                                                                                           \
        case 1: e = launch_kernel(k_search_topk<KSV, 1>, grid, kSrThreads, smem, st, s, R, E, tbl, ta, Kp, k, sel, part_v, part_i); break;   \
        case 2: e = launch_kernel(k_search_topk<KSV, 2>, grid, kSrThreads, smem, st, s, R, E, tbl, ta, Kp, k, sel, part_v, part_i); break;   \
        case 4: e = launch_kernel(k_search_topk<KSV, 4>, grid, kSrThreads, smem, st, s, R, E, tbl, ta, Kp, k, sel, part_v, part_i); break;   \
        case 8: e = launch_kernel(k_search_topk<KSV, 8>, grid, kSrThreads, smem, st, s, R, E, tbl, ta, Kp, k, sel, part_v, part_i); break;   \
        default: e = launch_kernel(k_search_topk<KSV, 16>, grid, kSrThreads, smem, st, s, R, E, tbl, ta, Kp, k, sel, part_v, part_i); break; \
    }
    switch (ks) {
        case 3: GPE_SR_KM(3) break;
        case 5: GPE_SR_KM(5) break;
        case 8: GPE_SR_KM(8) break;
        case 12: GPE_SR_KM(12) break;
        case 16: GPE_SR_KM(16) break;
        default: GPE_SR_KM(24) break;
    }
#undef GPE_SR_KM
    if (e != cudaSuccess || gy == 1) return e;
    const unsigned fg = grid_for(R, 128);
    switch (km) {
        case 1: return launch_kernel(k_search_merge<1>, fg, 128, 0, st, part_v, part_i, R, k, gy, sel);
        case 2: return launch_kernel(k_search_merge<2>, fg, 128, 0, st, part_v, part_i, R, k, gy, sel);
        case 4: return launch_kernel(k_search_merge<4>, fg, 128, 0, st, part_v, part_i, R, k, gy, sel);
        case 8: return launch_kernel(k_search_merge<8>, fg, 128, 0, st, part_v, part_i, R, k, gy, sel);
        default: return launch_kernel(k_search_merge<16>, fg, 128, 0, st, part_v, part_i, R, k, gy, sel);
    }
}

cudaError_t search_gather(const double* cand, int D, const int64_t* sel, int k, int j, int64_t R, double* x, cudaStream_t st) {
    return launch_kernel(k_search_gather, grid_for(R * D, 256), 256, 0, st, cand, D, sel, k, j, R, x);
}

cudaError_t search_output(const int64_t* sel, const double* cst, int64_t R, int k, int64_t* idx, double* cost, cudaStream_t st) {
    return launch_kernel(k_search_output, grid_for(R * k, 256), 256, 0, st, sel, cst, R, k, idx, cost);
}

}  // namespace gpe
