// Explicit instantiations of the fused predict kernels for one padded input dimension GPE_DP.
// Compiled once per DP (-DGPE_DP=..) so the variants build in parallel; see Makefile.
#include "predict_full.cuh"
#include "predict_mean.cuh"
#include "predict_bank_mean.cuh"
#include "predict_tiny.cuh"
#include "launch.h"
#include <stdio.h>
#include <stdlib.h>

#ifndef GPE_DP
#error "compile with -DGPE_DP=<padded input dimension>"
#endif

#define GPE_CAT2(a, b) a##b
#define GPE_CAT(a, b) GPE_CAT2(a, b)

namespace gpe {

// Template shape <MT, WR, WC, MINB, KB> of each fused configuration; nt_act in [nt_lo, nt_max] runs the instance with
// NT = nt_act, any other nt_act the nt_max instance with column predicates.  launch_full instantiates from this table and
// full_name reports from it.
struct FullShape { int MT, WR, WC, MINB, KB, nt_lo, nt_max; };
constexpr FullShape kShape[3] = {
    {4, 2, 4, 1, 2, 1, 8},    // cfg 0: TN = 64, Mp = 32 nt_act <= 256, 8 warps as 2 x 4, 1 CTA/SM
    {4, 1, 8, 1, 1, 5, 8},    // cfg 1: TN = 32, Mp = 64 nt_act <= 512, 8 warps as 1 x 8, 1 CTA/SM
    {2, 1, 8, 1, 1, 9, 16},   // cfg 2: TN = 16, Mp = 64 nt_act <= 1024, 8 warps as 1 x 8 (warp tile 16 x 128), 1 CTA/SM;
};                            //        also the small-batch plan

// EXACT: the caller guarantees p.nt_act == NT, so only the predicate-free (FULLNT) kernels are instantiated.  One
// instantiation per number of active column tiles: in a wider instantiation the guard `if (j >= nt_act) break` inside the
// unrolled DMMA loop keeps the B-fragment loads from being hoisted (measured: M = 200, nt_act = 7 of 8: 2.55e8 -> 3.0e8
// points/s; M = 100: 7.1e8 -> 7.9e8).  !EXACT (developer configurations, the small-batch plan): both kernels.
template <int CFG, int NT, bool EXACT>
static cudaError_t launch_cfg(const FullParams& p, int grid, size_t smem, cudaStream_t st) {
    constexpr int MT = kShape[CFG].MT, WR = kShape[CFG].WR, WC = kShape[CFG].WC, MINB = kShape[CFG].MINB, KB = kShape[CFG].KB;
    if (EXACT && p.nt_act != NT) return cudaErrorInvalidValue;
    auto kern = p.symmetric ? k_predict_full<MT, NT, WR, WC, GPE_DP, MINB, KB, true, true, false>
                            : k_predict_full<MT, NT, WR, WC, GPE_DP, MINB, KB, true, false, false>;
    if constexpr (!EXACT) {
        if (p.nt_act != NT)
            kern = p.symmetric ? k_predict_full<MT, NT, WR, WC, GPE_DP, MINB, KB, false, true, false>
                               : k_predict_full<MT, NT, WR, WC, GPE_DP, MINB, KB, false, false, false>;
    }
#if GPE_DP <= 16
    // fused Hessian variants (gpemu.cu only asks for them when the model is not symmetric-folded)
    if (p.hess != nullptr) {
        if (p.symmetric || MINB != 1 || WR * WC != 8) return cudaErrorInvalidValue;
        if constexpr (MINB == 1 && WR * WC == 8) {
            kern = k_predict_full<MT, NT, WR, WC, GPE_DP, MINB, KB, true, false, true>;
            if constexpr (!EXACT) {
                if (p.nt_act != NT) kern = k_predict_full<MT, NT, WR, WC, GPE_DP, MINB, KB, false, false, true>;
            }
        }
    }
#else
    if (p.hess != nullptr) return cudaErrorInvalidValue;
#endif
    return launch_kernel(kern, grid, WR * WC * 32, smem, st, p);
}

static cudaError_t launch_full(int cfg, const FullParams& p, int grid, size_t smem, cudaStream_t st) {
    switch (cfg) {
        case 0:
            switch (p.nt_act) {
                case 1: return launch_cfg<0, 1, true>(p, grid, smem, st);
                case 2: return launch_cfg<0, 2, true>(p, grid, smem, st);
                case 3: return launch_cfg<0, 3, true>(p, grid, smem, st);
                case 4: return launch_cfg<0, 4, true>(p, grid, smem, st);
                case 5: return launch_cfg<0, 5, true>(p, grid, smem, st);
                case 6: return launch_cfg<0, 6, true>(p, grid, smem, st);
                case 7: return launch_cfg<0, 7, true>(p, grid, smem, st);
                case 8: return launch_cfg<0, 8, true>(p, grid, smem, st);
                default: return cudaErrorInvalidValue;
            }
        case 1:
            switch (p.nt_act) {
                case 5: return launch_cfg<1, 5, true>(p, grid, smem, st);
                case 6: return launch_cfg<1, 6, true>(p, grid, smem, st);
                case 7: return launch_cfg<1, 7, true>(p, grid, smem, st);
                default: return launch_cfg<1, 8, false>(p, grid, smem, st);
            }
        case 2:
            switch (p.nt_act) {
                case 9: return launch_cfg<2, 9, true>(p, grid, smem, st);
                case 10: return launch_cfg<2, 10, true>(p, grid, smem, st);
                case 11: return launch_cfg<2, 11, true>(p, grid, smem, st);
                case 12: return launch_cfg<2, 12, true>(p, grid, smem, st);
                case 13: return launch_cfg<2, 13, true>(p, grid, smem, st);
                case 14: return launch_cfg<2, 14, true>(p, grid, smem, st);
                case 15: return launch_cfg<2, 15, true>(p, grid, smem, st);
                default: return launch_cfg<2, 16, false>(p, grid, smem, st);
            }
        default: return cudaErrorInvalidValue;
    }
}

static int full_name(int cfg, int nt_act, bool symmetric, char* buf, int len) {
    const FullShape& s = kShape[cfg];
    const int nt = nt_act >= s.nt_lo && nt_act <= s.nt_max ? nt_act : s.nt_max;
    return snprintf(buf, len, "k_predict_full<%d,%d,%d,%d,%d,%d,%d,%s,%s,false>", s.MT, nt, s.WR, s.WC, GPE_DP, s.MINB, s.KB,
                    nt == nt_act ? "true" : "false", symmetric ? "true" : "false");
}

// mean + gradient: the two-rows-per-thread kernel (k_predict_mean2) up to DP = 10 and at DP = 16; the one-row kernel
// (k_predict_mean) where two rows of test coordinates, differences and gradient sums no longer fit the register file
// (measured, tools/d_sweep_probe.py, M = 250: D = 12 9.3e8 vs 8.2e8 points/s, D = 16 7.5e8 vs 8.0e8, D = 24 5.1e8 vs
// 3.1e8, D = 32 3.6e8 vs 1.2e8).  GPE_MEAN_V1=1 / GPE_MEAN_V2=1 force one or the other.
static bool mean_v1() {
    static const bool v1 = getenv("GPE_MEAN_V1") != nullptr || ((GPE_DP == 12 || GPE_DP >= 24) && getenv("GPE_MEAN_V2") == nullptr);
    return v1;
}

static const char* mean_name() { return mean_v1() ? "k_predict_mean" : "k_predict_mean2"; }

static cudaError_t launch_mean(bool hess, const MeanParams& p, dim3 grid, size_t smem, cudaStream_t st) {
    if (p.smem_need == 0 || p.smem_need > smem) return cudaErrorInvalidConfiguration;   // carve-up vs launch (see MeanParams)
    if (hess) {
#if GPE_DP <= 12
        return launch_kernel(k_predict_mean<GPE_DP, true>, grid, kMeanThreads, smem, st, p);
#else
        // D > 12: row-block Hessian kernel (predict_mean.cuh::k_hessian_rows); mean / gradient, if also requested,
        // come from the plain mean kernel first
        if (p.mu != nullptr || p.deriv != nullptr) {
            MeanParams q = p;
            q.hess = nullptr;
            cudaError_t e = launch_kernel(k_predict_mean<GPE_DP, false>, grid, kMeanThreads, smem, st, q);
            if (e != cudaSuccess) return e;
        }
        constexpr int HR = (GPE_DP <= 16) ? 4 : 2;
        return launch_kernel(k_hessian_rows<GPE_DP, HR>, grid, kMeanThreads, smem, st, p);
#endif
    }
    auto kern = p.kstar != nullptr ? k_predict_mean2<GPE_DP, true>
                                   : (mean_v1() ? k_predict_mean<GPE_DP, false> : k_predict_mean2<GPE_DP, false>);
    return launch_kernel(kern, grid, kMeanThreads, smem, st, p);
}

template <int G, bool GRAD>
static cudaError_t launch_bank_g(const BankMeanParams& p, dim3 grid, size_t smem, cudaStream_t st) {
    return launch_kernel(k_bank_mean<GPE_DP, G, GRAD>, grid, kBankThreads, smem, st, p);
}

// group sizes per DP: launch.h::bank_group_ok
static cudaError_t launch_bank_mean(int G, bool grad, const BankMeanParams& p, dim3 grid, size_t smem, cudaStream_t st) {
    if (p.smem_need == 0 || p.smem_need > smem) return cudaErrorInvalidConfiguration;
#if GPE_DP <= 16
    if (!grad) {
        if (G == 4) return launch_bank_g<4, false>(p, grid, smem, st);
        if (G == 5) return launch_bank_g<5, false>(p, grid, smem, st);
        if (G == 8) return launch_bank_g<8, false>(p, grid, smem, st);
        if (G == 10) return launch_bank_g<10, false>(p, grid, smem, st);
        return cudaErrorInvalidValue;
    }
#endif
#if GPE_DP <= 10
    if (G == 3) return launch_bank_g<3, true>(p, grid, smem, st);
    if (G == 4) return launch_bank_g<4, true>(p, grid, smem, st);
    if (G == 5) return launch_bank_g<5, true>(p, grid, smem, st);
#elif GPE_DP == 12
    if (G == 3) return launch_bank_g<3, true>(p, grid, smem, st);
    if (G == 4) return launch_bank_g<4, true>(p, grid, smem, st);
#elif GPE_DP == 16
    if (G == 2) return launch_bank_g<2, true>(p, grid, smem, st);
    if (G == 3) return launch_bank_g<3, true>(p, grid, smem, st);
#endif
    return cudaErrorInvalidValue;
}

static cudaError_t launch_tiny(const TinyParams& p, int grid, size_t smem, cudaStream_t st) {
#if GPE_DP <= 16
    return launch_kernel(k_predict_tiny<GPE_DP>, grid, kTinyThreads, smem, st, p);   // cluster dimensions are part of the kernel
#else
    return cudaErrorInvalidValue;
#endif
}

extern const DpKernels GPE_CAT(kKernelsDp, GPE_DP) = {GPE_DP, launch_full, launch_mean, launch_bank_mean, launch_tiny, full_name, mean_name};

}  // namespace gpe
