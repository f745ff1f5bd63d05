// PCA back-projection: out (R, W) = A (R, E) . basis (E, W), A addressed with three strides.
//
//   fwd (N, W) = mu (N, E) . basis          -- the accumulation `fwd += pred_mu * basis_functions[i]` of
//                                              MultivariateEmulator.predict (gp_emulator/multivariate_gp.py:216), batched;
//   deriv_full (N, D, W) = sum_e deriv[n, e, d] basis[e, w]                                            (:218)
//
// A skinny FP64 GEMM (K = E <= 32) that sits on the FP64 ridge: 2 E W flop against 8 W bytes written per row (E = 20:
// 37 TFLOP/s of DMMA <-> 7.4 TB/s of output), so the tensor pipe AND the HBM write stream both have to stay busy.
// CTA = 64 rows, 8 warps as 2 (rows) x 4 (columns); a warp keeps its A fragments (32 rows x E) in registers for the
// whole sweep over W and produces 32 x 32 output tiles with DMMA.8x8x4.  The basis is pre-tiled at bank creation as
// [ks][Wp][4] (b_tiled[ks][w][c] = basis[4 ks + c][w], zero padded), the conflict-free B-fragment image the variance
// kernel uses, streamed in 128-column groups by TMA bulk copies through a two-stage mbarrier ring.  Two CTAs per SM.
//
// Two ways out of the SM:
//   k_project_tma  (default) the CTA stages a 64-row x 128-column tile in shared memory and ONE elected thread hands it to
//                  the TMA engine as two tensor-map stores (SASS UTMASTG): no LSU store instructions, no lg_throttle
//                  stalls -- the warps only issue DMMAs and st.shared while the copy engine drains the tile.  Output rows
//                  are W = 2101 doubles: only 8-byte aligned, and the row pitch (16,808 B) is not a multiple of 16, so no
//                  tensor map can describe the matrix directly.  PAIRS of rows are 16-byte aligned and 16 W bytes apart:
//                  the even rows are the tensor (W, R/2) with pitch 2 W, the odd rows live in the tensor (2 W, R/2) at
//                  column offset W; TMA clips the last column group (and the rows past R) against the tensor bounds by
//                  itself.  A box must START on a 16-byte boundary, though (an odd element coordinate is an illegal
//                  instruction -- found the hard way), and with W odd an odd row starts 8 bytes off: its 16-byte aligned
//                  columns are the odd ones.  So for odd W the odd rows' box is 126 columns wide and starts one column
//                  later, and the two columns per row and group that fall outside (the first and the last of the group)
//                  are written by the lanes that hold them, with plain stores.  Clipping, too, happens in 16-byte units:
//                  the even rows' tensor is declared W - 1 columns wide and their last column is a plain store as well.
//   k_project      the first version: per-warp smem transposition, then st.global of 256 contiguous bytes per instruction.
//                  Kept for outputs that are not 16-byte aligned, for slices that accumulate (banks of more than 32
//                  emulators) and for a handful of rows.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <mutex>

#include "gpe_math.cuh"
#include "gpe_ptx.cuh"
#include "launch.h"

namespace gpe {

constexpr int kProjThreads = 256, kProjRows = 64, kProjCols = 128;
constexpr int kProjPitch = 40;  // doubles; = 8 (mod 16) so a quarter-warp's 16-byte fragment stores hit 32 banks
template <int KS>   // k-steps of 4: E <= 4 KS
__global__ void __launch_bounds__(kProjThreads, 2) k_project(const double* __restrict__ A, int64_t R, int RD, int64_t ldn,
                                                             int64_t lde, int64_t ldd, const double* __restrict__ b_tiled,
                                                             int E, int W, int Wp, double* __restrict__ out, int accumulate) {
    extern __shared__ __align__(128) unsigned char psm[];
    uint64_t* full = reinterpret_cast<uint64_t*>(psm);          // [2]
    double* stage = reinterpret_cast<double*>(psm + 128);       // [2][KS][128][4]
    double* ctile = stage + 2 * (size_t)KS * kProjCols * 4;     // [8 warps][16][kProjPitch]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wr = warp >> 2, wc = warp & 3;
    smem_guard(128u + 2u * KS * kProjCols * 4u * 8u + 8u * 16u * kProjPitch * 8u);
    const int64_t r0 = (int64_t)blockIdx.x * kProjRows + wr * 32;
    const int ngroups = Wp / kProjCols;
    constexpr uint32_t ks_bytes = kProjCols * 4 * 8, stage_doubles = (uint32_t)KS * kProjCols * 4;
    if (tid == 0) {
        mbar_init(&full[0], 1);
        mbar_init(&full[1], 1);
        fence_mbar_init();
    }
    __syncthreads();
    auto load_group = [&](int g, int st) {   // thread 0
        mbar_arrive_expect_tx(&full[st], (uint32_t)KS * ks_bytes);
        for (int ks = 0; ks < KS; ++ks)
            tma_bulk_g2s(stage + (size_t)st * stage_doubles + (size_t)ks * kProjCols * 4,
                         b_tiled + ((size_t)ks * Wp + (size_t)g * kProjCols) * 4, ks_bytes, &full[st]);
    };
    // column groups g = blockIdx.y, blockIdx.y + gridDim.y, ...: with a handful of rows (the reference's one-point call:
    // 1 row of spectrum, D rows of Jacobian) the launcher spreads the W / 128 groups over gridDim.y CTAs instead of
    // walking them one after the other in a single CTA
    const int gy = (int)gridDim.y, g_first = (int)blockIdx.y;
    if (tid == 0) {
        if (g_first < ngroups) load_group(g_first, 0);
        if (g_first + gy < ngroups) load_group(g_first + gy, 1);
    }
    // A fragments: lane holds A[row = 8 i + lane / 4][k = 4 ks + lane % 4]
    double a[4][KS];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t r = r0 + 8 * i + (lane >> 2);
        const int64_t base = (r < R) ? (r / RD) * ldn + (r % RD) * ldd : 0;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
            const int e = 4 * ks + (lane & 3);
            a[i][ks] = (r < R && e < E) ? A[base + (int64_t)e * lde] : 0.0;
        }
    }
    const int nrow = (int)max((int64_t)0, min((int64_t)32, R - r0));
    double* ct = ctile + (size_t)warp * (16 * kProjPitch);
    uint32_t par = 0;
    for (int g = g_first, it = 0; g < ngroups; g += gy, ++it) {
        const int st = it & 1;
        mbar_wait(&full[st], (par >> st) & 1u);
        par ^= 1u << st;
        const double* bs = stage + (size_t)st * stage_doubles + (size_t)(wc * 32 + (lane >> 2)) * 4 + (lane & 3);
        double acc[4][4][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const double bf = bs[(size_t)ks * kProjCols * 4 + j * 32];
#pragma unroll
                for (int i = 0; i < 4; ++i) dmma_m8n8k4(acc[i][j][0], acc[i][j][1], a[i][ks], bf);
            }
        }
        const int w = g * kProjCols + wc * 32 + lane;
        double* o = out + r0 * W + w;
#pragma unroll
        for (int half = 0; half < 2; ++half) {   // rows 0..15, then 16..31 of the warp tile
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    *reinterpret_cast<double2*>(ct + (8 * i + (lane >> 2)) * kProjPitch + 8 * j + 2 * (lane & 3)) =
                        make_double2(acc[2 * half + i][j][0], acc[2 * half + i][j][1]);
            __syncwarp();
            if (w < W) {
#pragma unroll 4
                for (int rr = 0; rr < 16; ++rr)
                    if (16 * half + rr < nrow) {
                        double* q = o + (int64_t)(16 * half + rr) * W;
                        *q = accumulate ? *q + ct[rr * kProjPitch + lane] : ct[rr * kProjPitch + lane];   // (slices of E > 32)
                    }
            }
        }
        __syncthreads();   // every warp is done with this stage: refill it with group g + 2
        if (tid == 0 && g + 2 * gy < ngroups) load_group(g + 2 * gy, st);
    }
}

template <int KS>
cudaError_t launch_project(const double* A, int64_t R, int RD, int64_t ldn, int64_t lde, int64_t ldd,
                           const double* b_tiled, int E, int W, int Wp, double* out, int accumulate, cudaStream_t st) {
    const size_t psmem = 128 + 2 * (size_t)KS * kProjCols * 4 * 8 + 8 * 16 * kProjPitch * 8;
    // few row blocks: spread the column groups over gridDim.y so that about one wave of CTAs is in flight
    const int64_t nrb = (R + kProjRows - 1) / kProjRows;
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int gy = (int)std::max<int64_t>(1, std::min<int64_t>(Wp / kProjCols, (int64_t)sms / nrb));
    return launch_kernel(k_project<KS>, dim3((unsigned)nrb, (unsigned)gy), kProjThreads, psmem, st, A, R, RD, ldn, lde, ldd, b_tiled, E,
                         W, Wp, out, accumulate);
}

// ---- tensor-map variant ------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];\n" ::"l"(map),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory"); }

// WRG = row groups of 32 rows (4 warps each) per CTA.  WRG = 1: 128 threads, 32-row tiles, three co-resident CTAs per SM whose
// DMMA / staging / barrier phases drift apart (measured against WRG = 2, see DESIGN 4.3)
template <int KS, int WRG>   // k-steps of 4: E <= 4 KS
__global__ void __launch_bounds__(WRG * 128, (KS <= 5 ? (WRG == 1 ? 3 : 2) : 1)) k_project_tma(const double* __restrict__ A, int64_t R, int RD, int64_t ldn,
                                                                 int64_t lde, int64_t ldd, const double* __restrict__ b_tiled,
                                                                 int E, int W, int Wp,
                                                                 const __grid_constant__ CUtensorMap map_even,
                                                                 const __grid_constant__ CUtensorMap map_odd,
                                                                 double* __restrict__ out) {
    extern __shared__ __align__(128) unsigned char psm[];
    constexpr uint32_t stage_doubles = (uint32_t)KS * kProjCols * 4, ks_bytes = kProjCols * 4 * 8;
    uint64_t* full = reinterpret_cast<uint64_t*>(psm);          // [2]
    double* stage = reinterpret_cast<double*>(psm + 128);       // [2][KS][128][4]
    constexpr int kRows = WRG * 32, kPairs = WRG * 16;
    double* tile_even = stage + 2 * (size_t)stage_doubles;      // [kPairs row pairs][128]: rows 0, 2, 4, ... of the CTA tile
    double* tile_odd = tile_even + kPairs * kProjCols;          // [kPairs row pairs][128 - 2 shift]: rows 1, 3, 5, ...
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wr = warp >> 2, wc = warp & 3;
    smem_guard(128u + 2u * stage_doubles * 8u + 2u * kPairs * kProjCols * 8u);
    const int64_t r0 = (int64_t)blockIdx.x * kRows + wr * 32;
    const int ngroups = Wp / kProjCols;
    if (tid == 0) {
        mbar_init(&full[0], 1);
        mbar_init(&full[1], 1);
        fence_mbar_init();
    }
    __syncthreads();
    auto load_group = [&](int g, int st) {   // thread 0
        mbar_arrive_expect_tx(&full[st], (uint32_t)KS * ks_bytes);
        for (int ks = 0; ks < KS; ++ks)
            tma_bulk_g2s(stage + (size_t)st * stage_doubles + (size_t)ks * kProjCols * 4,
                         b_tiled + ((size_t)ks * Wp + (size_t)g * kProjCols) * 4, ks_bytes, &full[st]);
    };
    if (tid == 0) {
        load_group(0, 0);
        if (ngroups > 1) load_group(1, 1);
    }
    // A fragments: lane holds A[row = 8 i + lane / 4][k = 4 ks + lane % 4]
    double a[4][KS];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t r = r0 + 8 * i + (lane >> 2);
        const int64_t base = (r < R) ? (r / RD) * ldn + (r % RD) * ldd : 0;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
            const int e = 4 * ks + (lane & 3);
            a[i][ks] = (r < R && e < E) ? A[base + (int64_t)e * lde] : 0.0;
        }
    }
    // where this lane's C fragments go in the staged tile: row rl = 32 wr + 8 i + lane / 4 -> parity buffer, pair rl / 2.
    // shift = 1 (odd W): the odd-row tile holds columns [1, 127) of the group at pitch 126 (see the header comment)
    const int shift = W & 1, po = kProjCols - 2 * shift;
    const int rl0 = wr * 32 + (lane >> 2);
    const bool odd_row = rl0 & 1;
    const int cl0 = wc * 32 + 2 * (lane & 3);                    // this lane's first column inside the group (tile j = 0)
    double* const dst_even = tile_even + (size_t)(rl0 >> 1) * kProjCols + cl0;
    double* const dst_odd = tile_odd + (size_t)(rl0 >> 1) * po + cl0 - shift;
    const int pair0 = (int)(((int64_t)blockIdx.x * kRows) >> 1);
    uint32_t par = 0;
    for (int g = 0; g < ngroups; ++g) {
        const int st = g & 1;
        mbar_wait(&full[st], (par >> st) & 1u);
        par ^= 1u << st;
        const double* bs = stage + (size_t)st * stage_doubles + (size_t)(wc * 32 + (lane >> 2)) * 4 + (lane & 3);
        double acc[4][4][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const double bf = bs[(size_t)ks * kProjCols * 4 + j * 32];
#pragma unroll
                for (int i = 0; i < 4; ++i) dmma_m8n8k4(acc[i][j][0], acc[i][j][1], a[i][ks], bf);
            }
        }
        // the previous group's tile must have left shared memory (its TMA stores have finished READING it) and every
        // warp must be done with this basis stage before it is refilled
        if (tid == 0) tma_store_wait_read();
        __syncthreads();
        if (tid == 0 && g + 2 < ngroups) load_group(g + 2, st);
        if (!odd_row || shift == 0) {
            double* const d0 = odd_row ? dst_odd : dst_even;
            const int pitch4 = 4 * (odd_row ? po : kProjCols);
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    *reinterpret_cast<double2*>(d0 + (size_t)i * pitch4 + 8 * j) = make_double2(acc[i][j][0], acc[i][j][1]);
            if (shift && g == (W - 1) / kProjCols) {
                // odd W: the copy engine clips in 16-byte units, so the even rows' tensor ends at column W - 2 (an even
                // number of columns) and their last column is written here, by the lane that holds it
                const int jl = (W - 1) % kProjCols - cl0;        // 8 j for the owning lane (W - 1 is even, like cl0)
                if (jl >= 0 && jl < 32 && (jl & 7) == 0) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int64_t r = (int64_t)blockIdx.x * kRows + rl0 + 8 * i;
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            if (8 * j == jl && r < R) out[r * W + W - 1] = acc[i][j][0];
                    }
                }
            }
        } else {
            // odd row of an odd-W matrix: 8-byte stores into the shifted tile; the group's first and last column go
            // straight to global memory
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int64_t r = (int64_t)blockIdx.x * kRows + rl0 + 8 * i;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int cl = cl0 + 8 * j;
                    double* d = dst_odd + (size_t)i * 4 * po + 8 * j;
                    if (cl > 0) d[0] = acc[i][j][0];
                    else if (r < R) out[r * W + g * kProjCols] = acc[i][j][0];
                    if (cl + 1 < kProjCols - 1) d[1] = acc[i][j][1];
                    else if (r < R && g * kProjCols + cl + 1 < W) out[r * W + g * kProjCols + cl + 1] = acc[i][j][1];
                }
            }
        }
        fence_proxy_async();   // generic-proxy writes -> visible to the TMA (async proxy) read
        __syncthreads();
        if (tid == 0) {
            // even rows: tensor (W, ceil(R/2)); odd rows: tensor (2 W, floor(R/2)) at column offset W (+ 1 for odd W).
            // Columns past the end of a row and row pairs past R are clipped by the copy engine.
            tma_store_2d(&map_even, tile_even, g * kProjCols, pair0);
            tma_store_2d(&map_odd, tile_odd, W + g * kProjCols + shift, pair0);
            tma_store_commit();
        }
    }
    if (tid == 0) tma_store_wait_read();   // shared memory must outlive the last copy's reads
}

// ---- forward cost: the misfit of the back-projected spectra, reduced without materialising them ------------------
//   cost_n = 1/2 sum_w l_w (fwd_nw - obs_nw)^2,  grad_nd = sum_w l_w (fwd_nw - obs_nw) deriv_full_ndw
//          = sum_e deriv_ned s_ne  with  s (N, E) = u . basis^T,  u = l o (fwd - obs)           (multivariate_gp.py:216,218)
// CTA = 32 rows, 8 warps as 2 (16 rows) x 4 (32 columns of each 128-column group).  The basis streams through the
// two-stage TMA ring of k_project_tma; the fwd tile is formed by the same DMMA sequence as there (accumulators from
// zero, k-steps ascending; slices of 32 emulators each from zero, added in slice order), so an observation equal to the
// library's own fwd leaves a residual of exactly zero.  Residual and cost stay in registers.  The C fragment of u (lane:
// row lane / 4, columns 2 (lane % 4) + h) is the A operand of two k-steps of s = u . basis^T with k <-> column
// 2 (lane % 4) + h, B read from the staged basis group: no shared-memory round trip.  The four column warps add their
// partial s through shared memory once per row tile, in a fixed order.
//   KS: k-steps of 4 emulators per slice (4, 6 or 8; zero-padded emulators add exact zeros); nsl > 1: slices of 32
//   emulators (KS = 8), all staged per group; A fragments are then re-read per slice, and with GRAD the W sweep runs
//   once per slice of s (registers hold the s of one slice).
//   aux = [weights padded to Wp with zeros | shared observation padded to Wp], so the tail group adds exact zeros.
//   HESS (with GRAD): s itself goes to s_out (R, E) as well, the curvature coefficients of the cost's Hessian
//   (k_cost_hess); grad may then be NULL.
//   PW: per-point weights, row r of wts at r * w_ld, loaded beside the observations (zero past W) and used in place of
//   the weights in aux; the product l_rw r_rw is the same one, so rows equal to the shared weights give the same bits.
constexpr int kFcThreads = 256, kFcRows = 32, kFcPitch = 33;
template <int KS, bool GRAD, bool HESS, bool PW>
__device__ __forceinline__ void forward_cost_body(const double* __restrict__ mu, const double* __restrict__ deriv,
                                                  int64_t R, int E, int D, const double* __restrict__ obs,
                                                  int64_t obs_ld, const double* __restrict__ aux,
                                                  const double* __restrict__ b_tiled, int W, int Wp, int nsl,
                                                  double* __restrict__ cost, double* __restrict__ grad,
                                                  double* __restrict__ part, double* __restrict__ s_out,
                                                  const double* __restrict__ wts, int64_t w_ld) {
    extern __shared__ __align__(128) unsigned char psm[];
    constexpr int NT = KS / 2;                                   // n-tiles of 8 emulators per slice of s
    const int kstg = nsl == 1 ? KS : 8 * nsl;                    // k-steps staged per column group
    const uint32_t stage_doubles = (uint32_t)kstg * kProjCols * 4, ks_bytes = kProjCols * 4 * 8;
    uint64_t* full = reinterpret_cast<uint64_t*>(psm);           // [2]
    double* stage = reinterpret_cast<double*>(psm + 128);        // [2][kstg][128][4]
    double* red_s = stage + 2 * (size_t)stage_doubles;           // [4 column warps][32 rows][kFcPitch]
    double* red_c = red_s + 4 * kFcRows * kFcPitch;              // [4 column warps][32 rows]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wr = warp >> 2, wc = warp & 3;
    smem_guard(128u + 2u * stage_doubles * 8u + (4u * kFcRows * kFcPitch + 4u * kFcRows) * 8u);
    const int64_t t0 = (int64_t)blockIdx.x * kFcRows;
    // column groups y, y + gy, ... of this CTA (gy = gridDim.y > 1: a few rows, the groups spread over CTAs; the partial
    // sums go to `part` [gy][R][1 + E] and k_forward_cost_finish adds them in the order of y)
    const int gy = (int)gridDim.y, y0 = (int)blockIdx.y, ngroups = Wp / kProjCols;
    const int ng = (ngroups - y0 + gy - 1) / gy, nsweep = GRAD ? nsl : 1, nitems = nsweep * ng;
    if (tid == 0) {
        mbar_init(&full[0], 1);
        mbar_init(&full[1], 1);
        fence_mbar_init();
    }
    __syncthreads();
    auto load_item = [&](int it, int st) {   // thread 0: every staged k-step of the item's column group
        const int g = y0 + (it % ng) * gy;
        mbar_arrive_expect_tx(&full[st], (uint32_t)kstg * ks_bytes);
        for (int ks = 0; ks < kstg; ++ks)
            tma_bulk_g2s(stage + (size_t)st * stage_doubles + (size_t)ks * kProjCols * 4,
                         b_tiled + ((size_t)ks * Wp + (size_t)g * kProjCols) * 4, ks_bytes, &full[st]);
    };
    if (tid == 0) {
        load_item(0, 0);
        if (nitems > 1) load_item(1, 1);
    }
    // A fragments of slice sl: lane holds mu[row = 16 wr + 8 i + lane / 4][e = 32 sl + 4 ks + lane % 4]
    double a[2][KS];
    auto load_a = [&](int sl) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int64_t r = t0 + 16 * wr + 8 * i + (lane >> 2);
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
                const int e = 32 * sl + 4 * ks + (lane & 3);
                a[i][ks] = (r < R && e < E) ? mu[r * E + e] : 0.0;
            }
        }
    };
    if (nsl == 1) load_a(0);
    // observations of this lane's C-fragment elements: [i][j][h] = obs[row 16 wr + 8 i + lane / 4][column 8 j + 2 (lane % 4) + h
    // of the warp's 32], zero past W
    const double* obs1 = obs_ld == 0 ? aux + Wp : nullptr;
    double ob[2][4][2];
    double lw[2][4][2];                                          // PW: the weights of the same elements
    auto load_obs = [&](int g) {
        const int c0 = g * kProjCols + wc * 32 + 2 * (lane & 3);
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int64_t r = t0 + 16 * wr + 8 * i + (lane >> 2);
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int w = c0 + 8 * j + h;
                    ob[i][j][h] = obs1 ? obs1[w] : ((r < R && w < W) ? obs[r * obs_ld + w] : 0.0);
                    if (PW) lw[i][j][h] = (r < R && w < W) ? wts[r * w_ld + w] : 0.0;
                }
        }
    };
    load_obs(y0);
    double c[2] = {0.0, 0.0};                                    // per-lane share of sum u r of rows i
    double s[2][NT][2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) s[i][nt][0] = s[i][nt][1] = 0.0;
    uint32_t par = 0;
    for (int it = 0; it < nitems; ++it) {
        const int g = y0 + (it % ng) * gy, so = it / ng, st = it & 1;
        const bool last = it % ng == ng - 1;
        mbar_wait(&full[st], (par >> st) & 1u);
        par ^= 1u << st;
        const double* sb = stage + (size_t)st * stage_doubles;
        // 1. fwd tile of the warp: 16 rows x 32 columns
        double f[2][4][2];
        for (int sl = 0; sl < nsl; ++sl) {
            if (nsl > 1) load_a(sl);
            const double* bs = sb + (size_t)sl * 8 * kProjCols * 4 + (size_t)(wc * 32 + (lane >> 2)) * 4 + (lane & 3);
            double acc[2][4][2];
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const double bf = bs[(size_t)ks * kProjCols * 4 + j * 32];
#pragma unroll
                    for (int i = 0; i < 2; ++i) dmma_m8n8k4(acc[i][j][0], acc[i][j][1], a[i][ks], bf);
                }
            }
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int h = 0; h < 2; ++h) f[i][j][h] = sl == 0 ? acc[i][j][h] : f[i][j][h] + acc[i][j][h];
        }
        // 2. residual, weighted residual u (kept in f), cost
        const int c0 = g * kProjCols + wc * 32 + 2 * (lane & 3);
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const double r = f[i][j][h] - ob[i][j][h];
                    const double u = (PW ? lw[i][j][h] : aux[c0 + 8 * j + h]) * r;
                    if (so == 0) c[i] = fma(u, r, c[i]);
                    f[i][j][h] = u;
                }
        if (it + 1 < nitems) load_obs(y0 + ((it + 1) % ng) * gy);   // in flight during the s update and the next wait
        // 3. s (rows x emulators of slice so) += u . basis^T over this warp's 32 columns: 8 k-steps (j, h)
        if (GRAD) {
            const double* bsl = sb + (size_t)so * 8 * kProjCols * 4;
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int cl = wc * 32 + 8 * j + 2 * (lane & 3) + h;
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        // B[k = lane % 4][n = lane / 4] = basis[e = 8 nt + lane / 4][column cl]
                        const double bf = bsl[((size_t)(2 * nt + (lane >> 4)) * kProjCols + cl) * 4 + ((lane >> 2) & 3)];
#pragma unroll
                        for (int i = 0; i < 2; ++i) dmma_m8n8k4(s[i][nt][0], s[i][nt][1], f[i][j][h], bf);
                    }
                }
        }
        __syncthreads();   // every warp is done with this stage: refill it
        if (tid == 0 && it + 2 < nitems) load_item(it + 2, st);
        if (so == 0 && last) {
            // 4a. cost of the tile's rows: lanes of a row, then the four column warps, in a fixed order
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                double v = c[i] + __shfl_xor_sync(0xffffffffu, c[i], 1);
                v += __shfl_xor_sync(0xffffffffu, v, 2);
                if ((lane & 3) == 0) red_c[wc * kFcRows + 16 * wr + 8 * i + (lane >> 2)] = v;
            }
            __syncthreads();
            if (tid < kFcRows && t0 + tid < R) {
                const double v = ((red_c[tid] + red_c[kFcRows + tid]) + red_c[2 * kFcRows + tid]) + red_c[3 * kFcRows + tid];
                if (gy > 1) part[((size_t)y0 * R + t0 + tid) * (1 + E)] = v;
                else if (cost) cost[t0 + tid] = 0.5 * v;
            }
        }
        if (GRAD && last) {
            // 4b. grad_nd (+)= sum_{e in slice so} deriv_ned s_ne
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        red_s[(wc * kFcRows + 16 * wr + 8 * i + (lane >> 2)) * kFcPitch + 8 * nt + 2 * (lane & 3) + h] = s[i][nt][h];
                        s[i][nt][h] = 0.0;
                    }
            __syncthreads();
            const int es = min(32, E - 32 * so);
            for (int k = tid; k < kFcRows * es; k += kFcThreads) {
                const int rl = k / es, e = k - rl * es;
                double* q = red_s + rl * kFcPitch + e;
                *q = ((q[0] + q[kFcRows * kFcPitch]) + q[2 * kFcRows * kFcPitch]) + q[3 * kFcRows * kFcPitch];
            }
            __syncthreads();
            if (gy > 1) {
                for (int k = tid; k < kFcRows * es; k += kFcThreads) {
                    const int rl = k / es, e = k - rl * es;
                    if (t0 + rl < R) part[((size_t)y0 * R + t0 + rl) * (1 + E) + 1 + 32 * so + e] = red_s[rl * kFcPitch + e];
                }
            } else if (HESS) {
                for (int k = tid; k < kFcRows * es; k += kFcThreads) {
                    const int rl = k / es, e = k - rl * es;
                    if (t0 + rl < R) s_out[(t0 + rl) * E + 32 * so + e] = red_s[rl * kFcPitch + e];
                }
            }
            for (int k = tid; k < kFcRows * D && gy == 1 && (!HESS || grad); k += kFcThreads) {
                const int rl = k / D, d = k - rl * D;
                const int64_t r = t0 + rl;
                if (r >= R) continue;
                const double* dp = deriv + (r * E + 32 * so) * D + d;
                double v = 0.0;
                for (int e = 0; e < es; ++e) v = fma(dp[(size_t)e * D], red_s[rl * kFcPitch + e], v);
                grad[r * D + d] = so == 0 ? v : grad[r * D + d] + v;
            }
            __syncthreads();   // red_s is rewritten by the next sweep
        }
    }
}

template <int KS, bool GRAD, bool HESS>
__global__ void __launch_bounds__(kFcThreads, 1) k_forward_cost(const double* __restrict__ mu, const double* __restrict__ deriv,
                                                                int64_t R, int E, int D, const double* __restrict__ obs,
                                                                int64_t obs_ld, const double* __restrict__ aux,
                                                                const double* __restrict__ b_tiled, int W, int Wp, int nsl,
                                                                double* __restrict__ cost, double* __restrict__ grad,
                                                                double* __restrict__ part, double* __restrict__ s_out) {
    forward_cost_body<KS, GRAD, HESS, false>(mu, deriv, R, E, D, obs, obs_ld, aux, b_tiled, W, Wp, nsl, cost, grad, part, s_out,
                                             nullptr, 0);
}

// Per-point weights (DESIGN 4.6f): wts (R, w_ld), l_rw = wts[r * w_ld + w].
template <int KS, bool GRAD, bool HESS>
__global__ void __launch_bounds__(kFcThreads, 1) k_forward_cost_pw(const double* __restrict__ mu, const double* __restrict__ deriv,
                                                                   int64_t R, int E, int D, const double* __restrict__ obs,
                                                                   int64_t obs_ld, const double* __restrict__ aux,
                                                                   const double* __restrict__ b_tiled, int W, int Wp, int nsl,
                                                                   double* __restrict__ cost, double* __restrict__ grad,
                                                                   double* __restrict__ part, double* __restrict__ s_out,
                                                                   const double* __restrict__ wts, int64_t w_ld) {
    forward_cost_body<KS, GRAD, HESS, true>(mu, deriv, R, E, D, obs, obs_ld, aux, b_tiled, W, Wp, nsl, cost, grad, part, s_out,
                                            wts, w_ld);
}

// aux = [weights or 1, zero past W | shared observation, zero past W] (one launch per call)
__global__ void k_forward_cost_aux(const double* __restrict__ weights, const double* __restrict__ obs1, int W, int Wp,
                                   double* __restrict__ aux) {
    for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < Wp; w += gridDim.x * blockDim.x) {
        aux[w] = w < W ? (weights ? weights[w] : 1.0) : 0.0;
        if (obs1) aux[Wp + w] = w < W ? obs1[w] : 0.0;
    }
}

// C (E, E) = basis . diag(l) . basis^T, the Gauss-Newton operand of the forward cost's Hessian (k_cost_hess), from the
// tiled basis image and the padded weights in aux (one launch per call).  One warp per entry e <= f: lanes stride over
// w, then a fixed butterfly; the entry is written to (e, f) and (f, e), so C is exactly symmetric.
__global__ void k_forward_cost_curv(const double* __restrict__ b_tiled, const double* __restrict__ aux, int E, int Wp,
                                    double* __restrict__ C) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; k < (int64_t)E * E; k += nwarps) {
        const int e = (int)(k / E), f = (int)(k - (int64_t)e * E);
        if (f < e) continue;
        const double* be = b_tiled + (size_t)(e >> 2) * Wp * 4 + (e & 3);
        const double* bf = b_tiled + (size_t)(f >> 2) * Wp * 4 + (f & 3);
        double v = 0.0;
        for (int w = lane; w < Wp; w += 32) v = fma(be[(size_t)4 * w] * aux[w], bf[(size_t)4 * w], v);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) C[(int64_t)e * E + f] = C[(int64_t)f * E + e] = v;
    }
}

// Per-point curvature (DESIGN 4.6f): C_n (E, E) = basis . diag(l_n) . basis^T for the rows l_n = wts[n * w_ld + .] (zero past
// W), summed exactly as k_forward_cost_curv sums C: lane L adds fma(b_ew l_nw, b_fw, v) over w = L, L + 32, ... < Wp in
// order, then the same xor butterfly, so a row equal to the shared weights gives the shared C bit for bit.  One warp
// takes a 4 x 4 tile of entries (e in block a, f in block c >= a) of one point: every lane keeps 16 sums, and per w it
// loads l once and the two 4-wide basis columns once.  Consecutive warps take the same tile of consecutive points, so a
// CTA reads each basis column from L1 for 8 points.  Entries e <= f < E are written to (e, f) and (f, e).
__global__ void __launch_bounds__(256) k_forward_cost_curv_pw(const double* __restrict__ b_tiled, const double* __restrict__ wts,
                                                              int64_t w_ld, int64_t n, int E, int W, int Wp,
                                                              double* __restrict__ C) {
    const int lane = threadIdx.x & 31, nb = (E + 3) / 4, ntile = nb * (nb + 1) / 2;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; k < n * ntile; k += nwarps) {
        const int t = (int)(k / n);
        const int64_t p = k - (int64_t)t * n;
        int a = 0, q = t;
        while (q >= nb - a) { q -= nb - a; ++a; }
        const int c = a + q;
        const double* ba = b_tiled + (size_t)a * Wp * 4;
        const double* bc = b_tiled + (size_t)c * Wp * 4;
        const double* l = wts + p * w_ld;
        double v[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) v[i][j] = 0.0;
        for (int w = lane; w < Wp; w += 32) {
            const double lw = w < W ? l[w] : 0.0;
            const double2 e01 = *reinterpret_cast<const double2*>(ba + 4 * (size_t)w);
            const double2 e23 = *reinterpret_cast<const double2*>(ba + 4 * (size_t)w + 2);
            const double2 f01 = *reinterpret_cast<const double2*>(bc + 4 * (size_t)w);
            const double2 f23 = *reinterpret_cast<const double2*>(bc + 4 * (size_t)w + 2);
            const double be[4] = {e01.x * lw, e01.y * lw, e23.x * lw, e23.y * lw}, bf[4] = {f01.x, f01.y, f23.x, f23.y};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) v[i][j] = fma(be[i], bf[j], v[i][j]);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v[i][j] += __shfl_xor_sync(0xffffffffu, v[i][j], o);
            }
        if (lane < 16) {
            double out = 0.0;
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) if (lane == 4 * i + j) out = v[i][j];
            const int e = 4 * a + (lane >> 2), f = 4 * c + (lane & 3);
            if (e <= f && f < E) {
                double* Cp = C + p * E * E;
                Cp[(int64_t)e * E + f] = Cp[(int64_t)f * E + e] = out;
            }
        }
    }
}

// Column-split calls: cost_r = 1/2 sum_y part[y][r][0], s_re = sum_y part[y][r][1 + e], grad_rd = sum_e deriv_red s_re
// (HESS: s also to s_out (R, E), by the threads of d = 0)
template <bool HESS>
__global__ void k_forward_cost_finish(const double* __restrict__ part, const double* __restrict__ deriv, int64_t R, int E, int D,
                                      int gy, double* __restrict__ cost, double* __restrict__ grad, double* __restrict__ s_out) {
    const int64_t pitch = (int64_t)R * (1 + E);
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < R * (D + 1); k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = k / (D + 1);
        const int d = (int)(k - r * (D + 1)) - 1;               // -1: the cost
        const double* p = part + r * (1 + E);
        if (d < 0) {
            double v = 0.0;
            for (int y = 0; y < gy; ++y) v += p[y * pitch];
            if (cost) cost[r] = 0.5 * v;
        } else if (grad || HESS) {
            double v = 0.0;
            for (int e = 0; e < E; ++e) {
                double se = 0.0;
                for (int y = 0; y < gy; ++y) se += p[y * pitch + 1 + e];
                if (HESS && d == 0) s_out[r * E + e] = se;
                v = fma(deriv[(r * E + e) * D + d], se, v);
            }
            if (grad) grad[r * D + d] = v;
        }
    }
}

int forward_cost_split(int64_t call_N, int W) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int64_t tiles = (call_N + kFcRows - 1) / kFcRows, ngroups = (W + kProjCols - 1) / kProjCols;
    return (int)std::max<int64_t>(1, std::min<int64_t>(ngroups, (int64_t)sms / tiles));
}

size_t forward_cost_smem(int E) {
    const int nsl = (E + 31) / 32, ks = (E + 3) / 4;
    const int kstg = nsl == 1 ? (ks <= 4 ? 4 : ks <= 6 ? 6 : 8) : 8 * nsl;
    return 128 + 2 * (size_t)kstg * kProjCols * 4 * 8 + (4 * (size_t)kFcRows * kFcPitch + 4 * kFcRows) * 8;
}

cudaError_t forward_cost_aux(const double* weights, const double* obs1, int W, int Wp, double* aux, cudaStream_t st) {
    return launch_kernel(k_forward_cost_aux, (unsigned)((Wp + 255) / 256), 256, 0, st, weights, obs1, W, Wp, aux);
}

cudaError_t forward_cost_curv(const double* b_tiled, const double* aux, int E, int Wp, double* C, cudaStream_t st) {
    const int64_t warps = (int64_t)E * E;
    return launch_kernel(k_forward_cost_curv, (unsigned)std::min<int64_t>((warps + 7) / 8, 4096), 256, 0, st, b_tiled, aux, E, Wp, C);
}

cudaError_t forward_cost_curv_pw(const double* b_tiled, const double* wts, int64_t w_ld, int64_t n, int E, int W, int Wp, double* C,
                                cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    const int nb = (E + 3) / 4;
    const int64_t warps = n * (nb * (nb + 1) / 2);
    return launch_kernel(k_forward_cost_curv_pw, (unsigned)std::min<int64_t>((warps + 7) / 8, (int64_t)148 * 64), 256, 0, st,
                         b_tiled, wts, w_ld, n, E, W, Wp, C);
}

cudaError_t forward_cost_rows(const double* mu, const double* deriv, int64_t R, int E, int D, const double* obs, int64_t obs_ld,
                              const double* aux, const double* b_tiled, int W, int Wp, int gy, double* part, double* cost,
                              double* grad, double* s_out, cudaStream_t st, const double* wts, int64_t w_ld) {
    const int nsl = (E + 31) / 32, ks = (E + 3) / 4;
    const size_t smem = forward_cost_smem(E);
    const dim3 grid((unsigned)((R + kFcRows - 1) / kFcRows), (unsigned)gy);
    cudaError_t e;
#define GPE_FC(KSV)                                                                                                          \
    e = s_out ? launch_kernel(k_forward_cost<KSV, true, true>, grid, kFcThreads, smem, st, mu, deriv, R, E, D, obs, obs_ld,   \
                              aux, b_tiled, W, Wp, nsl, cost, grad, part, s_out)                                             \
        : grad ? launch_kernel(k_forward_cost<KSV, true, false>, grid, kFcThreads, smem, st, mu, deriv, R, E, D, obs, obs_ld, \
                               aux, b_tiled, W, Wp, nsl, cost, grad, part, s_out)                                            \
               : launch_kernel(k_forward_cost<KSV, false, false>, grid, kFcThreads, smem, st, mu, deriv, R, E, D, obs,       \
                               obs_ld, aux, b_tiled, W, Wp, nsl, cost, grad, part, s_out)
#define GPE_FC_PW(KSV)                                                                                                       \
    e = s_out ? launch_kernel(k_forward_cost_pw<KSV, true, true>, grid, kFcThreads, smem, st, mu, deriv, R, E, D, obs,        \
                              obs_ld, aux, b_tiled, W, Wp, nsl, cost, grad, part, s_out, wts, w_ld)                          \
        : grad ? launch_kernel(k_forward_cost_pw<KSV, true, false>, grid, kFcThreads, smem, st, mu, deriv, R, E, D, obs,      \
                               obs_ld, aux, b_tiled, W, Wp, nsl, cost, grad, part, s_out, wts, w_ld)                         \
               : launch_kernel(k_forward_cost_pw<KSV, false, false>, grid, kFcThreads, smem, st, mu, deriv, R, E, D, obs,    \
                               obs_ld, aux, b_tiled, W, Wp, nsl, cost, grad, part, s_out, wts, w_ld)
    if (w_ld != 0) {
        if (nsl == 1 && ks <= 4) GPE_FC_PW(4);
        else if (nsl == 1 && ks <= 6) GPE_FC_PW(6);
        else GPE_FC_PW(8);
    } else {
        if (nsl == 1 && ks <= 4) GPE_FC(4);
        else if (nsl == 1 && ks <= 6) GPE_FC(6);
        else GPE_FC(8);
    }
#undef GPE_FC
#undef GPE_FC_PW
    if (e != cudaSuccess || gy == 1) return e;
    const unsigned fgrid = (unsigned)((R * (D + 1) + 127) / 128);
    return s_out ? launch_kernel(k_forward_cost_finish<true>, fgrid, 128, 0, st, part, deriv, R, E, D, gy, cost, grad, s_out)
                 : launch_kernel(k_forward_cost_finish<false>, fgrid, 128, 0, st, part, deriv, R, E, D, gy, cost, grad, s_out);
}

namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// cuTensorMapEncodeTiled through the runtime (libcuda is not linked): resolved once.
EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            p = nullptr;
        }
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// Tensor maps of the even and the odd output rows (see the header comment).  false: not expressible -> LSU kernel.
bool make_row_pair_maps(double* out, int64_t R, int W, int pairs, CUtensorMap* even, CUtensorMap* odd) {
    EncodeTiledFn enc = encode_tiled();
    if (!enc || (reinterpret_cast<uintptr_t>(out) & 15) != 0 || R < 2) return false;
    const cuuint64_t pitch[1] = {(cuuint64_t)W * 16};           // two rows, in bytes: a multiple of 16 for any W
    const cuuint32_t box[2] = {(cuuint32_t)kProjCols, (cuuint32_t)pairs}, estr[2] = {1, 1};
    const cuuint32_t box_odd[2] = {(cuuint32_t)(kProjCols - 2 * (W & 1)), (cuuint32_t)pairs};   // odd W: see the header comment
    // (odd W: W - 1 columns -- the engine clips in 16-byte units; the kernel writes the even rows' last column itself)
    const cuuint64_t dim_even[2] = {(cuuint64_t)(W - (W & 1)), (cuuint64_t)((R + 1) / 2)};
    const cuuint64_t dim_odd[2] = {(cuuint64_t)2 * W, (cuuint64_t)(R / 2)};
    if (enc(even, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, out, dim_even, pitch, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return false;
    if (enc(odd, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, out, dim_odd, pitch, box_odd, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return false;
    return true;
}

template <int KS, int WRG>
cudaError_t launch_project_tma(const double* A, int64_t R, int RD, int64_t ldn, int64_t lde, int64_t ldd, const double* b_tiled,
                               int E, int W, int Wp, const CUtensorMap& even, const CUtensorMap& odd, double* out, cudaStream_t st) {
    const size_t psmem = 128 + 2 * (size_t)KS * kProjCols * 4 * 8 + 2 * (size_t)WRG * 16 * kProjCols * 8;
    return launch_kernel(k_project_tma<KS, WRG>, (unsigned)((R + WRG * 32 - 1) / (WRG * 32)), WRG * 128, psmem, st, A, R, RD, ldn, lde,
                         ldd, b_tiled, E, W, Wp, even, odd, out);
}

}  // namespace

cudaError_t project_rows(const double* A, int64_t R, int RD, int64_t ldn, int64_t lde, int64_t ldd, const double* b_tiled, int E,
                         int W, int Wp, double* out, int accumulate, cudaStream_t st) {
    static const bool no_tma = getenv("GPE_PROJECT_NO_TMA") != nullptr;   // dev aid: time / test the LSU kernel
    const int ks = (E + 3) / 4;
    CUtensorMap even, odd;
    static const int wrg = getenv("GPE_PROJECT_WR") ? atoi(getenv("GPE_PROJECT_WR")) : 1;   // dev aid: 2 = 64-row CTAs
    // (a few rows -- the reference's one-point call -- keep the LSU kernel: its stores may go straight to mapped host memory)
    if (!accumulate && !no_tma && R >= 256 && make_row_pair_maps(out, R, W, wrg == 2 ? 32 : 16, &even, &odd)) {
#define GPE_PROJ_TMA(KSV)                                                                                                   \
        return wrg == 2 ? launch_project_tma<KSV, 2>(A, R, RD, ldn, lde, ldd, b_tiled, E, W, Wp, even, odd, out, st)     \
                        : launch_project_tma<KSV, 1>(A, R, RD, ldn, lde, ldd, b_tiled, E, W, Wp, even, odd, out, st)
        if (ks <= 3) GPE_PROJ_TMA(3);
        if (ks <= 5) GPE_PROJ_TMA(5);
        GPE_PROJ_TMA(8);
#undef GPE_PROJ_TMA
    }
    if (ks <= 3) return launch_project<3>(A, R, RD, ldn, lde, ldd, b_tiled, E, W, Wp, out, accumulate, st);
    if (ks <= 5) return launch_project<5>(A, R, RD, ldn, lde, ldd, b_tiled, E, W, Wp, out, accumulate, st);
    return launch_project<8>(A, R, RD, ldn, lde, ldd, b_tiled, E, W, Wp, out, accumulate, st);
}

}  // namespace gpe
