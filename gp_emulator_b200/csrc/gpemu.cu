// libgpemu.so -- C ABI implementation (see include/gpemu.h for the contract and reference citations).
//
// Host responsibilities: validate, lay the trained model out for the kernels (done once per model, the
// reference re-uploads and re-transposes it for every 2e5-point block: gp_emulator/gpu/predict.cu:11-34,
// _gpu_predict.cpp:129-132), pick the kernel configuration, launch, and -- for host-resident callers --
// stream test points through a two-slot pinned pipeline (replaces the Python chunk loop of
// GaussianProcess.gpu_predict / get_gpu_block, gp_emulator/GaussianProcess.py:253-323).
#include <cuda_runtime.h>
#include <pthread.h>
#include <sched.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <cmath>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/gpemu.h"
#include "launch.h"
#include "predict_generic.cuh"
#include "gpe_math.cuh"
#include "host_common.h"
#include "host_stream.h"

using namespace gpe;

namespace {

thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};
long long* g_trace = nullptr;  // dev aid: device buffer for per-tile phase timestamps (gpe_debug_trace)

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess)                                                                           \
            return fail(GPE_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

constexpr uint32_t kSmemMax = 232448;  // 227 KB opt-in limit per CTA on sm_100
inline uint32_t align_up(uint32_t x, uint32_t a) { return (x + a - 1) / a * a; }

constexpr int kHessFusedMaxDp = 16;   // predict_full_inst.cu instantiates the HESS variants up to this DP

struct FullPlan {
    bool valid = false;
    int cfg = 0, TN = 0, WC = 0, GH = 1, ctas_per_sm = 1;
    int Mp = 0, nt_act = 0, kblk = 0, kbps = 0, nit = 0, nstage = 0, JC = 0, nchunks = 0;
    uint32_t off_bar = 0, off_sqw = 0, off_ks = 0, off_bst = 0, off_xc = 0, off_ts = 0, off_pa = 0, off_vred = 0;
    uint32_t stage_bytes = 0, smem = 0, ts_bytes = 0;
    // fused Hessian (phase C of the fused kernel): P operand width, k-blocks per ring stage, iterations
    uint32_t off_hts = 0;
    int NC = 0, kbh = 0, nit_h = 0;
};

struct Tf32Plan {
    bool valid = false;
    int DP = 0, Mp = 0, nslab = 0;
    bool big = false;      // 256 < M <= 1024: column passes + A ring (predict_tf32_big.cuh)
    int pass_cols = 0;
    uint32_t off_bar = 0, off_tmem = 0, off_a = 0, off_b = 0, off_x = 0, off_out = 0, off_vred = 0, bstage_bytes = 0, smem = 0;
};

struct MeanPlan {
    int JC = 0, nchunks = 0;
    uint32_t off_xc = 0, off_ts = 0, off_out = 0, smem = 0, smem_hess = 0;
};

// Shared-difference bank kernel (predict_bank_mean.cuh): groups of G emulators per thread
struct BankMeanPlan {
    bool valid = false;
    int G = 0, ngroups = 0, JC = 0, nchunks = 0;
    uint32_t off_x = 0, off_a = 0, off_w = 0, off_ts = 0, smem = 0;
};

}  // namespace

struct gpe_model {
    int device = 0, M = 0, D = 0, DP = 0, sms = 0;
    double b = 0;
    double sqrt_w[32];
    bool has_invQ = false;
    bool symmetric = false;      // GPE_OPT_SYMMETRIC_VARIANCE: s_tiled holds the upper-triangular fold of invQ
    FullPlan full;
    FullPlan full_small;         // 16-point tiles for small batches (valid only if it can share the main plan's operands)
    MeanPlan mean;
    double* d_xchunks_full = nullptr;
    double* d_stiled = nullptr;
    double* d_ptiled = nullptr;  // Hessian operand of the fused kernel (null: direct Hessian kernel only)
    // 1024 < M <= GPE_MAX_TRAIN: two-launch variance path (predict_var_large.cuh); d_stiled then has Mp / 4 k-blocks
    bool large_valid = false;
    int large_Mp = 0, large_kblk = 0, large_nstage = 0;
    int64_t large_chunk = 0;             // points per sub-batch = capacity of the K* scratch
    double* d_kscratch = nullptr;        // [large_chunk / 16][large_kblk][16][4], pads stay zero
    cudaEvent_t scratch_free = nullptr;  // the scratch is shared by every stream that predicts with this model
    std::mutex scratch_mu;               // wait -> launches -> record on the scratch is one critical section per caller
    double centre[32];
    bool hess_fused_ok = false;
    double* d_xchunks_mean = nullptr;
    // D > 32: generic kernels (predict_generic.cuh) + the large-M variance kernel on the same K* scratch
    bool generic = false;
    double* d_gen_xs = nullptr;     // (M, D) inputs scaled by sqrt(w)
    double* d_gen_alpha = nullptr;  // (M) b * invQt
    double* d_gen_sqw = nullptr;    // (D)
    double* d_gen_mu = nullptr;     // (large_chunk) means of the sub-batch in flight
    Tf32Plan tf, tfx;            // single-precision tcgen05 paths: fast (1 x TF32) and precise (3 x TF32); lazy
    float* d_xa_f32 = nullptr;
    uint32_t* d_bslabs = nullptr;
    uint32_t* d_bslabs_lo = nullptr;
    std::vector<double> h_inputs, h_invQt, h_invQ;  // host copy of the model for the lazy FP32 packing
    double h_expx[33];
    std::mutex host_mu;          // host-pointer calls on one model share its slots (and the lazy FP32 packing): one at a time
    Slot slots[3];               // host-streaming pipeline: the direct (pinned caller) path uses two, the staged path three
};

struct gpe_bank {
    int device = 0, E = 0, M = 0, D = 0, W = 0;
    std::vector<gpe_model*> models;
    MeanBankEntry* d_entries = nullptr;  // per-emulator phase-A data for the one-launch bank mean / Hessian kernel
    // shared input differences (k_bank_mean), when compiled for (DP, G): [1] mean + gradient, [0] means only (larger groups)
    BankMeanPlan gplan[2];
    double* d_gx = nullptr;              // raw training inputs [nchunks][JC][DP]
    double* d_galpha[2] = {nullptr, nullptr};   // [ngroups][nchunks][JC][GP]
    double* d_gw[2] = {nullptr, nullptr};       // [ngroups][2][G][DP]
    double* d_basis = nullptr;   // basis pre-tiled as [ks][Wp][4] per slice of 32 emulators, Wp = W rounded up to 128
    int Wp = 0;
    // host-pointer calls (GPE_HOST_PTRS, gpe_bank_forward): the bank's own streaming slots, one call at a time
    std::mutex host_mu;
    Slot slots[3];
    double* d_aux = nullptr;     // shared observation vector + weights of a host-pointer gpe_bank_cost call
    size_t aux_cap = 0;
    // gpe_bank_cost: per-chunk mu / deriv scratch, shared by every stream that reduces with this bank
    std::mutex cost_mu;
    double* cost_d = nullptr;
    size_t cost_cap = 0;
    cudaEvent_t cost_free = nullptr;
};

struct gpe_multi {
    std::vector<int> devices;
    std::vector<gpe_model*> models;   // one resident copy of the GP per device (single-GP handle) ...
    std::vector<gpe_bank*> banks;     // ... or of the bank (bank handle)
    // PCIe routing of host-resident calls: relays[g].partner >= 0 sends device g's host traffic through that device's
    // link over NVLink (decided once per handle from a measured link rate, multi_route)
    std::mutex route_mu;
    bool routed = false;
    std::vector<Relay> relays;
    std::vector<double> link_gbs;     // measured per-device rate (GB/s per direction, all devices copying both ways at once)
};

namespace {

int pick_dp(int D) {
    for (int i = 0; i < kNumDp; ++i)
        if (kDpList[i] >= D) return kDpList[i];
    return -1;
}

cudaError_t launch_full(int DP, int cfg, const FullParams& p, int grid, size_t smem, cudaStream_t st) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    switch (DP) {
        case 2: return launch_full_dp2(cfg, p, grid, smem, st);
        case 4: return launch_full_dp4(cfg, p, grid, smem, st);
        case 6: return launch_full_dp6(cfg, p, grid, smem, st);
        case 8: return launch_full_dp8(cfg, p, grid, smem, st);
        case 10: return launch_full_dp10(cfg, p, grid, smem, st);
        case 12: return launch_full_dp12(cfg, p, grid, smem, st);
        case 16: return launch_full_dp16(cfg, p, grid, smem, st);
        case 24: return launch_full_dp24(cfg, p, grid, smem, st);
        case 32: return launch_full_dp32(cfg, p, grid, smem, st);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_mean(int DP, bool hess, const MeanParams& p, dim3 grid, size_t smem, cudaStream_t st) {
    if (p.smem_need == 0 || p.smem_need > smem) return cudaErrorInvalidConfiguration;   // carve-up vs launch (see MeanParams)
    g_launches.fetch_add(1, std::memory_order_relaxed);
    switch (DP) {
        case 2: return launch_mean_dp2(hess, p, grid, smem, st);
        case 4: return launch_mean_dp4(hess, p, grid, smem, st);
        case 6: return launch_mean_dp6(hess, p, grid, smem, st);
        case 8: return launch_mean_dp8(hess, p, grid, smem, st);
        case 10: return launch_mean_dp10(hess, p, grid, smem, st);
        case 12: return launch_mean_dp12(hess, p, grid, smem, st);
        case 16: return launch_mean_dp16(hess, p, grid, smem, st);
        case 24: return launch_mean_dp24(hess, p, grid, smem, st);
        case 32: return launch_mean_dp32(hess, p, grid, smem, st);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_tiny(int DP, const TinyParams& p, int grid, size_t smem, cudaStream_t st) {
    switch (DP) {
        case 2: return launch_tiny_dp2(p, grid, smem, st);
        case 4: return launch_tiny_dp4(p, grid, smem, st);
        case 6: return launch_tiny_dp6(p, grid, smem, st);
        case 8: return launch_tiny_dp8(p, grid, smem, st);
        case 10: return launch_tiny_dp10(p, grid, smem, st);
        case 12: return launch_tiny_dp12(p, grid, smem, st);
        case 16: return launch_tiny_dp16(p, grid, smem, st);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_bank_mean(int DP, int G, bool grad, const BankMeanParams& p, dim3 grid, size_t smem, cudaStream_t st) {
    if (p.smem_need == 0 || p.smem_need > smem) return cudaErrorInvalidConfiguration;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    switch (DP) {
        case 2: return launch_bank_mean_dp2(G, grad, p, grid, smem, st);
        case 4: return launch_bank_mean_dp4(G, grad, p, grid, smem, st);
        case 6: return launch_bank_mean_dp6(G, grad, p, grid, smem, st);
        case 8: return launch_bank_mean_dp8(G, grad, p, grid, smem, st);
        case 10: return launch_bank_mean_dp10(G, grad, p, grid, smem, st);
        case 12: return launch_bank_mean_dp12(G, grad, p, grid, smem, st);
        case 16: return launch_bank_mean_dp16(G, grad, p, grid, smem, st);
        default: return cudaErrorInvalidValue;
    }
}

// Group size and shared-memory carve-up of k_bank_mean for a bank of E emulators: the G that minimises the FP64
// instruction count  ceil(E / G) (G (2D + 12) + 2D)  (means only: G (D + 11) + 2D) among the compiled ones; invalid when
// none is compiled for DP or the one-emulator kernels (E (3D + 13)) would not be slower.
BankMeanPlan plan_bank_mean(int E, int M, int D, int DP, bool grad) {
    BankMeanPlan g;
    long best = (long)E * (3 * D + 13);
    const int per_em = grad ? 2 * D + 12 : D + 11;
    for (int G = 2; G <= 10; ++G) {
        if (!bank_group_ok(DP, G, grad)) continue;
        const long cost = (long)((E + G - 1) / G) * (G * per_em + 2 * D);
        if (cost < best) { best = cost; g.G = G; }
    }
    if (const char* e = getenv(grad ? "GPE_BANK_G" : "GPE_BANK_G_MEAN"))   // developer aid: force a group size
        if (bank_group_ok(DP, atoi(e), grad)) g.G = atoi(e);
    if (g.G == 0) return g;
    const int GP = (g.G + 1) & ~1;
    g.ngroups = (E + g.G - 1) / g.G;
    const int m4 = (M + 3) / 4 * 4;
    g.JC = std::min(m4, 256);
    g.nchunks = (M + g.JC - 1) / g.JC;
    uint32_t off = 0;
    g.off_x = off; off += align_up((uint32_t)g.JC * x_pitch(DP) * 8u, 16);
    g.off_a = off; off += align_up((uint32_t)g.JC * GP * 8u, 16);
    g.off_w = off; off += align_up(2u * g.G * DP * 8u, 16);
    g.off_ts = off; off += align_up((uint32_t)kBankTN * (uint32_t)std::max(D, g.G * (grad ? DP + 1 : 1)) * 8u, 16);
    g.smem = off;
    g.valid = true;
    return g;
}

// Decide tile shape, pipeline depth and the shared-memory carve-up of the fused kernel for (M, D).
//   cfg 0: Mp <= 256 -> TN = 64, 8 warps as 2 x 4, 1 CTA/SM
//   cfg 1 / 2: Mp <= 512 / 1024, TN = 32 / 16, 8 warps as 1 x 8, 1 CTA/SM
// (Two more configurations were measured and dropped in round 1: two co-resident 4-warp CTAs per SM -- slower, mixing
// DFMA and DMMA warps costs pipe efficiency and per-tile overheads double -- and 16 warps at 128 registers, which spills.)
// small_Mp > 0: the low-latency plan for small batches -- 16-point tiles (cfg 2) on the padded width of the main
// plan, so that both share s_tiled / xchunks.
FullPlan plan_full(int M, int D, int DP, int small_Mp = 0) {
    FullPlan f;
    const int m32 = (M + 31) / 32 * 32, m64 = (M + 63) / 64 * 64;
    // the kernels also hold static shared memory (exp table 512 B; HESS variants a 1 KB index table + 256 B): leave room
    const uint32_t smem_cap = kSmemMax - 2048;
    if (small_Mp > 0) {
        f.cfg = 2; f.TN = 16; f.WC = 8; f.GH = 4; f.Mp = small_Mp; f.nt_act = small_Mp / 64;
    } else if (m32 <= 256) {
        f.cfg = 0; f.TN = 64; f.WC = 4; f.GH = 1; f.Mp = m32; f.nt_act = m32 / 32;
    } else if (m64 <= 512) {
        f.cfg = 1; f.TN = 32; f.WC = 8; f.GH = 2; f.Mp = m64; f.nt_act = m64 / 64;
    } else if (m64 <= 1024) {
        f.cfg = 2; f.TN = 16; f.WC = 8; f.GH = 4; f.Mp = m64; f.nt_act = m64 / 64;
    } else {
        return f;  // invalid: variance contraction unsupported for this M
    }
    f.ctas_per_sm = 1;
    f.kblk = (M + 3) / 4;
    f.kbps = (f.cfg == 0) ? 2 : 1;  // k-blocks (32 * Mp bytes each) per ring stage == template KB of the cfg
    f.nit = (f.kblk + f.kbps - 1) / f.kbps;
    f.stage_bytes = (uint32_t)f.kbps * f.Mp * 32u;

    uint32_t off = 0;
    f.off_bar = off; off += 192;
    f.off_sqw = off; off += 256;
    f.off_ks = off; off += (uint32_t)f.TN * (f.Mp + 4) * 8u;
    f.ts_bytes = align_up((uint32_t)f.TN * (D + 1) * 8u, 16);  // x2: current rows / output staging + prefetch
    f.off_ts = off; off += 2 * f.ts_bytes;
    f.off_pa = off; off += (f.GH > 1) ? align_up((uint32_t)f.GH * f.TN * (D + 1) * 8u, 16) : 0;
    f.off_vred = off; off += (uint32_t)f.WC * f.TN * 8u;
    if (DP <= kHessFusedMaxDp) {   // room for the centred test rows of the fused Hessian
        f.off_hts = off; off += align_up((uint32_t)f.TN * D * 8u, 16);
        f.NC = (DP * (DP + 1) / 2 + 7) / 8 * 8;
        f.kbh = (int)(f.stage_bytes / ((uint32_t)f.NC * 32u));
        f.nit_h = f.kbh > 0 ? (f.kblk + f.kbh - 1) / f.kbh : 0;
    }
    off = align_up(off, 128);
    const uint32_t fixed = off;
    const int m4 = (M + 3) / 4 * 4;
    const uint32_t row = (uint32_t)(x_pitch(DP) + 1) * 8u;
    // resident training set if it fits beside a ring of >= 3 stages, else chunks of <= 256 points; the ring then
    // takes every stage that still fits (at most 8: the barrier arrays)
    {
        const uint32_t avail = smem_cap - fixed;
        const uint32_t resident = (uint32_t)m4 * row;
        if (avail >= resident + 3 * f.stage_bytes) {
            f.JC = m4; f.nchunks = 1;
        } else {
            if (avail < 2 * f.stage_bytes + 64 * row) return f;
            const int jc_max = (int)((avail - 2 * f.stage_bytes) / row) / 4 * 4;
            f.JC = std::min(std::min(jc_max, 256), m4); f.nchunks = (M + f.JC - 1) / f.JC;
        }
        f.nstage = (int)std::min<uint32_t>(8, (avail - (uint32_t)f.JC * row) / f.stage_bytes);
        if (f.nstage < 2) return f;
    }
    f.off_bst = fixed;
    f.off_xc = fixed + (uint32_t)f.nstage * f.stage_bytes;
    f.smem = f.off_xc + (uint32_t)f.JC * row;
    f.valid = f.smem <= smem_cap;
    return f;
}

MeanPlan plan_mean(int M, int D, int DP) {
    MeanPlan m;
    const int m4 = (M + 3) / 4 * 4;
    m.JC = std::min(m4, 256);
    m.nchunks = (M + m.JC - 1) / m.JC;
    uint32_t off = 0;
    m.off_xc = off; off += align_up((uint32_t)m.JC * (x_pitch(DP) + 1) * 8u, 16);
    m.off_ts = off; off += align_up((uint32_t)kMeanTN * (D + 1) * 8u, 16);
    m.off_out = off;
    m.smem = off;
    // Hessian staging: [TN][D][D] for the triangular kernel (D <= 12), [TN][HR][D] for the row-block kernel
    m.smem_hess = off + (uint32_t)kMeanTN * D * 8u * (uint32_t)(DP <= 12 ? D : (DP <= 16 ? 4 : 2));
    return m;
}

// Extent of the mean kernels' shared-memory carve-up, recomputed from the offsets the kernels use (checked against the
// dynamic shared memory of the launch at kernel entry: MeanParams::smem_need).
uint32_t mean_extent(const MeanPlan& mp, int D, int DP, bool hess) {
    uint32_t ext = std::max(mp.off_xc + (uint32_t)mp.JC * (x_pitch(DP) + 1) * 8u, mp.off_ts + (uint32_t)kMeanTN * (D + 1) * 8u);
    if (hess) ext = std::max(ext, mp.off_out + (uint32_t)kMeanTN * D * 8u * (uint32_t)(DP <= 12 ? D : (DP <= 16 ? 4 : 2)));
    return ext;
}

// [nchunks][ JC*DP sqrt(w)-scaled inputs | JC b*alpha ], zero padded
std::vector<double> pack_xchunks(int M, int D, int DP, int JC, int nchunks, const double* inputs,
                                 const double* sqrt_w, const double* invQt, double b) {
    const int XP = x_pitch(DP);   // row pitch: conflict-free LDS.128 in the kernels (gpe_math.cuh)
    std::vector<double> buf((size_t)nchunks * JC * (XP + 1), 0.0);
    for (int j = 0; j < M; ++j) {
        const int c = j / JC, jl = j - c * JC;
        double* base = buf.data() + (size_t)c * JC * (XP + 1);
        for (int d = 0; d < D; ++d) base[(size_t)jl * XP + d] = sqrt_w[d] * inputs[(size_t)j * D + d];
        base[(size_t)JC * XP + jl] = b * invQt[j];
    }
    return buf;
}

int check_device(int device, int* sms) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(GPE_ERR_NO_DEVICE, "no CUDA device available (%s); libgpemu has no CPU fallback",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(GPE_ERR_INVALID, "device %d out of range [0, %d)", device, n);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(GPE_ERR_NO_DEVICE, "device %d is sm_%d%d; libgpemu kernels are built for sm_100a only", device,
                    prop.major, prop.minor);
    *sms = prop.multiProcessorCount;
    return GPE_OK;
}

// Operand of the fused Hessian (predict_full.cuh, phase C): p_tiled[kb][col][c] = b alpha_j x'_jd x'_je for
// j = 4 kb + c, col = index of (d <= e) in the row-major upper triangle, x' = sqrt(w) x - centre (mid-range).
// The expansion sum k a (x'_d - t'_d)(x'_e - t'_e) = S2 - t'_d g_e - t'_e g_d - t'_d t'_e S0 loses about
// log10(max |x'|^2) digits to cancellation, so it is only enabled while max |x'|^2 <= kHessFusedMaxR2
// (training inputs within ~45 length scales of the centre: error amplification <= 2e3 * 2^-53 ~ 2e-13);
// beyond that, and for the shapes the fused kernel does not cover, the direct kernel runs.
constexpr double kHessFusedMaxR2 = 2000.0;

int build_hessian_operand(gpe_model* m, const double* inputs, const double* invQt) {
    const FullPlan& f = m->full;
    const int M = m->M, D = m->D;
    memset(m->centre, 0, sizeof(m->centre));
    m->hess_fused_ok = false;
    if (getenv("GPE_HESS_DIRECT") != nullptr) return GPE_OK;   // dev aid: always use the direct Hessian kernels
    if (!f.valid || f.kbh < 1 || f.NC > M || f.NC > f.Mp) return GPE_OK;
    double r2max = 0.0;
    for (int d = 0; d < D; ++d) {
        double lo = inputs[d], hi = inputs[d];
        for (int j = 1; j < M; ++j) { lo = std::min(lo, inputs[(size_t)j * D + d]); hi = std::max(hi, inputs[(size_t)j * D + d]); }
        m->centre[d] = m->sqrt_w[d] * 0.5 * (lo + hi);
        const double r = m->sqrt_w[d] * 0.5 * (hi - lo);
        r2max = std::max(r2max, r * r);
    }
    if (!(r2max <= kHessFusedMaxR2)) return GPE_OK;
    std::vector<double> pt((size_t)f.kblk * f.NC * 4, 0.0);
    std::vector<double> xp(D);
    for (int j = 0; j < M; ++j) {
        for (int d = 0; d < D; ++d) xp[d] = m->sqrt_w[d] * inputs[(size_t)j * D + d] - m->centre[d];
        const double ba = m->b * invQt[j];
        int col = 0;
        for (int d = 0; d < D; ++d)
            for (int e = d; e < D; ++e, ++col) pt[((size_t)(j >> 2) * f.NC + col) * 4 + (j & 3)] = ba * xp[d] * xp[e];
    }
    cudaError_t e = cudaMalloc((void**)&m->d_ptiled, pt.size() * 8);
    if (e == cudaSuccess) e = cudaMemcpy(m->d_ptiled, pt.data(), pt.size() * 8, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return fail(GPE_ERR_CUDA, "model upload failed: %s", cudaGetErrorString(e));
    m->hess_fused_ok = true;
    return GPE_OK;
}

// D > 32 (predict_generic.cuh): K* of a sub-batch into the model's scratch, then gradient / variance / Hessian from it.
int predict_generic(gpe_model* m, const double* testing, int64_t N, double* mu, double* var, double* deriv, double* hess,
                    int64_t ld_mu, int64_t ld_var, int64_t ld_deriv, int64_t ld_hess, cudaStream_t st) {
    if (var != nullptr && !m->has_invQ) return fail(GPE_ERR_INVALID, "variance requested but the model was created without invQ");
    if (var != nullptr && !m->large_valid)
        return fail(GPE_ERR_UNSUPPORTED, "variance contraction supports M <= %d (got M = %d)", GPE_MAX_TRAIN, m->M);
    const int D = m->D;
    const size_t smem_k = ((size_t)(kGenTN + kGenJC) * (D + 1) + 128) * 8;
    CUDA_TRY(cudaFuncSetAttribute(k_generic_kstar, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_k));
    std::lock_guard<std::mutex> scratch_lock(m->scratch_mu);   // one caller at a time between wait and record (see below)
    CUDA_TRY(cudaStreamWaitEvent(st, m->scratch_free, 0));
    for (int64_t n0 = 0; n0 < N; n0 += m->large_chunk) {
        const int64_t n = std::min(m->large_chunk, N - n0);
        GenericParams p;
        memset(&p, 0, sizeof(p));
        p.testing = testing + n0 * D; p.N = n;
        p.mu = mu ? mu + n0 * ld_mu : nullptr;
        p.deriv = deriv ? deriv + n0 * ld_deriv : nullptr;
        p.hess = hess ? hess + n0 * ld_hess : nullptr;
        p.ld_mu = ld_mu; p.ld_deriv = ld_deriv; p.ld_hess = ld_hess;
        p.xs = m->d_gen_xs; p.alpha = m->d_gen_alpha; p.sqw = m->d_gen_sqw;
        p.kstar = m->d_kscratch; p.mu_tmp = m->d_gen_mu;
        p.M = m->M; p.D = D; p.kblk = m->large_kblk;
        const int64_t tiles = (n + kGenTN - 1) / kGenTN;
        g_launches.fetch_add(1, std::memory_order_relaxed);
        k_generic_kstar<<<(unsigned)std::min<int64_t>(tiles, (int64_t)m->sms * 4), kGenThreads, smem_k, st>>>(p);
        CUDA_TRY(cudaGetLastError());
        if (deriv != nullptr) {
            g_launches.fetch_add(1, std::memory_order_relaxed);
            k_generic_grad<<<dim3((unsigned)std::min<int64_t>(tiles, (int64_t)m->sms * 8), (unsigned)std::min((D + 15) / 16, 16)),
                             kGenThreads, 0, st>>>(p);
            CUDA_TRY(cudaGetLastError());
        }
        if (var != nullptr) {
            VarLargeParams v;
            memset(&v, 0, sizeof(v));
            v.kstar = m->d_kscratch; v.s_tiled = m->d_stiled; v.var = var + n0 * ld_var; v.ld_var = ld_var; v.N = n;
            v.Mp = m->large_Mp; v.kblk = m->large_kblk; v.npass = (m->large_Mp + kVlPass - 1) / kVlPass;
            v.nstage = m->large_nstage; v.b = m->b;
            const size_t smem = 128 + kVlWarps * kVlTN * 8 + (size_t)v.nstage * kVlStageBytes;
            g_launches.fetch_add(1, std::memory_order_relaxed);
            CUDA_TRY(launch_var_large(v, (int)std::min<int64_t>((n + kVlTN - 1) / kVlTN, m->sms), smem, st));
        }
        if (hess != nullptr) {
            g_launches.fetch_add(1, std::memory_order_relaxed);
            k_generic_hess<<<(unsigned)std::min<int64_t>(n, (int64_t)m->sms * 8), kGenThreads, 0, st>>>(p);
            CUDA_TRY(cudaGetLastError());
        }
    }
    CUDA_TRY(cudaEventRecord(m->scratch_free, st));
    return GPE_OK;
}

// Whether a mean + variance + gradient call of call_N points takes the cluster path (predict_tiny.cuh): the fused plan's
// resident training chunk, a compiled DP, and few enough points (GPE_TINY_MAX overrides the threshold, GPE_NO_TINY disables).
bool tiny_ok(const gpe_model* m, int64_t call_N) {
    static const bool no_tiny = getenv("GPE_NO_TINY") != nullptr;
    static const int64_t env_max = getenv("GPE_TINY_MAX") ? atoll(getenv("GPE_TINY_MAX")) : -1;
    // two clusters per 8 SMs: measured at M = 250 (tools/tiny_threshold_probe.py, synchronous device calls) the cluster path
    // takes 37.9 us against 49.3 us at 500 points and draws level with the 16-point plan at 1000
    const int64_t n_max = env_max >= 0 ? env_max : kTinyTN * (int64_t)(2 * m->sms / kTinyCluster);
    return !no_tiny && m->full.valid && m->full.cfg == 0 && m->full.nchunks == 1 && m->DP <= 16 && call_N <= n_max;
}

// Launch the kernels for device-resident data on `st`.  Output strides allow bank (point-major) layouts.
int predict_device(gpe_model* m, const double* testing, int64_t N, double* mu, double* var, double* deriv,
                   double* hess, int64_t ld_mu, int64_t ld_var, int64_t ld_deriv, int64_t ld_hess,
                   cudaStream_t st, int64_t call_N = -1) {
    // call_N: size of the API call this launch is a chunk of (the host pipeline); plan choices that change the
    // summation order depend on it, not on the chunk, so that one call is internally consistent
    if (call_N < 0) call_N = N;
    if (N == 0) return GPE_OK;
    if (m->generic) return predict_generic(m, testing, N, mu, var, deriv, hess, ld_mu, ld_var, ld_deriv, ld_hess, st);
    bool mean_done = false;
    static const bool force_full = getenv("GPE_FORCE_FULL") != nullptr;  // dev aid: time phase A alone
    // the Hessian rides on the fused kernel when the model qualifies (build_hessian_operand); without a variance
    // request that only pays for the 64-point tiles of cfg 0 (measured: 4.6e8 vs 3.6e8 points/s at M = 250, but
    // 0.98e8 vs 1.10e8 at M = 1000), so larger M keeps the direct kernel for Hessian-only calls
    // (the HESS variants are built on the plain variance operand: with a symmetric-folded model the Hessian only rides
    // along when no variance is requested -- phase B is then skipped and the fold does not matter)
    // (calls small enough for the cluster path below take the variance from it whatever else is requested, and the Hessian
    // from the direct kernel: every output of a call of a given size comes from the same kernel for any combination of flags)
    const bool tiny = m->has_invQ && tiny_ok(m, call_N);
    const bool fuse_hess = hess != nullptr && m->hess_fused_ok && !tiny && (var != nullptr ? !m->symmetric : m->full.cfg == 0);
    if (var != nullptr && m->has_invQ && !m->full.valid && m->large_valid) {
        // 1024 < M <= GPE_MAX_TRAIN: per sub-batch, K* + mean + gradient (k_predict_mean2<DP, true>) into the scratch,
        // then the column-pass contraction (k_var_large).  The scratch is per model: streams take turns.
        // (two threads on different streams must not both pass the wait before either records: hold the model's
        // scratch mutex from the wait to the record, as gpe_bank_cost does for its scratch)
        std::lock_guard<std::mutex> scratch_lock(m->scratch_mu);
        CUDA_TRY(cudaStreamWaitEvent(st, m->scratch_free, 0));
        for (int64_t n0 = 0; n0 < N; n0 += m->large_chunk) {
            const int64_t n = std::min(m->large_chunk, N - n0);
            MeanParams p;
            memset(&p, 0, sizeof(p));
            p.testing = testing + n0 * m->D; p.N = n;
            p.mu = mu ? mu + n0 * ld_mu : nullptr;
            p.deriv = deriv ? deriv + n0 * ld_deriv : nullptr;
            p.ld_mu = ld_mu; p.ld_deriv = ld_deriv;
            p.xchunks = m->d_xchunks_mean; p.M = m->M; p.D = m->D; p.JC = m->mean.JC; p.nchunks = m->mean.nchunks;
            p.off_xc = m->mean.off_xc; p.off_ts = m->mean.off_ts; p.off_out = m->mean.off_out;
            p.smem_need = mean_extent(m->mean, m->D, m->DP, false);
            p.kstar = m->d_kscratch; p.kblk = m->large_kblk;
            memcpy(p.sqrt_w, m->sqrt_w, sizeof(p.sqrt_w));
            const int64_t mtiles = (n + kMeanTN - 1) / kMeanTN;
            CUDA_TRY(launch_mean(m->DP, false, p, dim3((unsigned)std::min<int64_t>(mtiles, (int64_t)m->sms * 12)), m->mean.smem, st));
            VarLargeParams v;
            memset(&v, 0, sizeof(v));
            v.kstar = m->d_kscratch; v.s_tiled = m->d_stiled; v.var = var + n0 * ld_var; v.ld_var = ld_var; v.N = n;
            v.Mp = m->large_Mp; v.kblk = m->large_kblk; v.npass = (m->large_Mp + kVlPass - 1) / kVlPass;
            v.nstage = m->large_nstage; v.b = m->b;
            const size_t smem = 128 + kVlWarps * kVlTN * 8 + (size_t)v.nstage * kVlStageBytes;
            const int64_t vtiles = (n + kVlTN - 1) / kVlTN;
            g_launches.fetch_add(1, std::memory_order_relaxed);
            CUDA_TRY(launch_var_large(v, (int)std::min<int64_t>(vtiles, m->sms), smem, st));
        }
        CUDA_TRY(cudaEventRecord(m->scratch_free, st));
        mean_done = true;
        var = nullptr;
    }
    // A handful of points (up to two clusters per 8 SMs): the latency path, one 8-CTA cluster per 16-point tile
    // (predict_tiny.cuh).  Needs the fused plan's resident training chunk; a Hessian request goes the usual way.
    if (var != nullptr && tiny) {
        const FullPlan& f = m->full;
        TinyParams p;
        memset(&p, 0, sizeof(p));
        p.testing = testing; p.N = N; p.mu = mu; p.var = var; p.deriv = deriv;
        p.ld_mu = ld_mu; p.ld_var = ld_var; p.ld_deriv = ld_deriv;
        p.xchunks = m->d_xchunks_full; p.s_tiled = m->d_stiled;
        p.M = m->M; p.D = m->D; p.JC = f.JC; p.Mp = f.Mp; p.kblk = f.kblk; p.b = m->b;
        memcpy(p.sqrt_w, m->sqrt_w, sizeof(p.sqrt_w));
        const size_t work = std::max<size_t>({(size_t)f.JC * (x_pitch(m->DP) + 1) + (size_t)kTinyTN * m->D,
                                              (size_t)16 * 16 * (m->DP + 1), (size_t)8 * 16 * 32});
        const size_t smem = ((size_t)kTinyTN * (f.Mp + 4) + work) * 8;
        const int grid = (int)((N + kTinyTN - 1) / kTinyTN) * kTinyCluster;
        g_launches.fetch_add(1, std::memory_order_relaxed);
        CUDA_TRY(launch_tiny(m->DP, p, grid, smem, st));
        mean_done = true;
        var = nullptr;
    }
    if (var != nullptr || fuse_hess || (force_full && m->full.valid)) {
        if (var != nullptr && !m->has_invQ) return fail(GPE_ERR_INVALID, "variance requested but the model was created without invQ");
        if (!m->full.valid)
            return fail(GPE_ERR_UNSUPPORTED, "variance contraction supports M <= %d (got M = %d)", GPE_MAX_TRAIN, m->M);
        // up to three waves of 16-point tiles finish sooner than one wave of 64-point tiles
        const bool small = m->full_small.valid && !fuse_hess && call_N <= 3 * 16 * (int64_t)m->sms;
        const FullPlan& f = small ? m->full_small : m->full;
        FullParams p;
        memset(&p, 0, sizeof(p));
        p.testing = testing; p.N = N; p.mu = mu; p.var = var; p.deriv = deriv;
        p.ld_mu = ld_mu; p.ld_var = ld_var; p.ld_deriv = ld_deriv;
        p.xchunks = m->d_xchunks_full; p.s_tiled = m->d_stiled;
        p.M = m->M; p.D = m->D; p.Mp = f.Mp; p.nt_act = f.nt_act; p.kblk = f.kblk;
        p.nit = f.nit; p.nstage = f.nstage; p.lag = (f.nstage >= 3) ? 2 : 1; p.symmetric = (m->symmetric && var != nullptr) ? 1 : 0;
        if (const char* e = getenv("GPE_RING_LAG")) p.lag = std::max(1, std::min(atoi(e), f.nstage - 1));
        // 64-point tiles, full width (Mp = 256): the second warp of every sub-partition starts its ring steps ~300 cycles
        // late (measured: M = 250 2.170e8 -> 2.193e8 points/s for 200 ... 600 cycles, M = 256 +1 %; neutral for narrower
        // tiles, -3 % at M = 32, nothing for the 16-point tiles of M = 1000: tools/m_sweep_probe.py, GPE_SKEW)
        p.skew = (f.cfg == 0 && f.nt_act == 8) ? 300 : 0;
        if (const char* e = getenv("GPE_SKEW")) p.skew = atoi(e);
        p.JC = f.JC; p.nchunks = f.nchunks; p.b = m->b;
        p.off_bar = f.off_bar; p.off_sqw = f.off_sqw; p.off_ks = f.off_ks; p.off_bst = f.off_bst;
        p.off_xc = f.off_xc; p.off_ts = f.off_ts; p.off_pa = f.off_pa; p.off_vred = f.off_vred;
        p.stage_bytes = f.stage_bytes; p.ts_bytes = f.ts_bytes;
        memcpy(p.sqrt_w, m->sqrt_w, sizeof(p.sqrt_w));
        p.trace = g_trace;
        if (fuse_hess) {
            p.hess = hess; p.ld_hess = ld_hess; p.p_tiled = m->d_ptiled; p.kbh = f.kbh; p.nit_h = f.nit_h; p.off_hts = f.off_hts;
            memcpy(p.centre, m->centre, sizeof(p.centre));
            hess = nullptr;   // done by this launch
        }
        const int64_t ntiles = (N + f.TN - 1) / f.TN;
        const int grid = (int)std::min<int64_t>(ntiles, (int64_t)m->sms * f.ctas_per_sm);
        CUDA_TRY(launch_full(m->DP, f.cfg, p, grid, f.smem, st));
        mean_done = true;
    }
    const bool need_mean = !mean_done && (mu != nullptr || deriv != nullptr);
    if (need_mean || hess != nullptr) {
        const bool do_hess = hess != nullptr;
        MeanParams p;
        memset(&p, 0, sizeof(p));
        p.testing = testing; p.N = N;
        p.mu = mean_done ? nullptr : mu;
        p.deriv = mean_done ? nullptr : deriv;
        p.hess = hess;
        p.ld_mu = ld_mu; p.ld_deriv = ld_deriv; p.ld_hess = ld_hess;
        p.xchunks = m->d_xchunks_mean; p.M = m->M; p.D = m->D; p.JC = m->mean.JC; p.nchunks = m->mean.nchunks;
        p.off_xc = m->mean.off_xc; p.off_ts = m->mean.off_ts; p.off_out = m->mean.off_out;
        p.smem_need = mean_extent(m->mean, m->D, m->DP, do_hess);
        memcpy(p.sqrt_w, m->sqrt_w, sizeof(p.sqrt_w));
        const int64_t ntiles = (N + kMeanTN - 1) / kMeanTN;
        // CTAs per SM: a multiple of what is resident (3 for the mean + gradient kernel, 2 / 4 for the Hessian ones)
        static const int env_mult = getenv("GPE_MEAN_GRID") ? atoi(getenv("GPE_MEAN_GRID")) : 0;
        const int mult = env_mult > 0 ? env_mult : (do_hess ? 8 : 12);
        const int grid = (int)std::min<int64_t>(ntiles, (int64_t)m->sms * mult);
        const size_t smem = do_hess ? m->mean.smem_hess : m->mean.smem;
        CUDA_TRY(launch_mean(m->DP, do_hess, p, dim3(grid), smem, st));
    }
    return GPE_OK;
}

// Calls that visit several devices leave the caller's current device as they found it (torch allocates on it).
struct DeviceRestore {
    int dev = -1;
    DeviceRestore() { if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); dev = -1; } }
    ~DeviceRestore() { if (dev >= 0) cudaSetDevice(dev); }
};

struct IoList {
    IoSpec v[kMaxIo];
    int n = 0;
    int add(const void* host, int64_t width) {
        if (n >= kMaxIo) return -1;
        v[n].host = const_cast<void*>(host);
        v[n].width = width;
        return n++;
    }
};

// Pin the calling thread to the CPUs that are local to `device` (sysfs local_cpulist of its PCI function), so that the
// staging copies and first touches of a per-device pipeline thread stay on the GPU's NUMA node.  Best effort.
void bind_thread_near_device(int device) {
    char bdf[32];
    if (cudaDeviceGetPCIBusId(bdf, sizeof(bdf), device) != cudaSuccess) { cudaGetLastError(); return; }
    for (char* c = bdf; *c; ++c) *c = (char)tolower(*c);
    const std::string path = std::string("/sys/bus/pci/devices/") + bdf + "/local_cpulist";
    FILE* f = fopen(path.c_str(), "r");
    if (!f) return;
    char line[4096];
    cpu_set_t set;
    CPU_ZERO(&set);
    int count = 0;
    if (fgets(line, sizeof(line), f)) {
        char* save = nullptr;
        for (char* tok = strtok_r(line, ",\n", &save); tok; tok = strtok_r(nullptr, ",\n", &save)) {
            int a = 0, b = 0;
            if (sscanf(tok, "%d-%d", &a, &b) == 2) { for (int i = a; i <= b && i < CPU_SETSIZE; ++i) { CPU_SET(i, &set); ++count; } }
            else if (sscanf(tok, "%d", &a) == 1 && a < CPU_SETSIZE) { CPU_SET(a, &set); ++count; }
        }
    }
    fclose(f);
    if (count > 0) pthread_setaffinity_np(pthread_self(), sizeof(set), &set);
}

// Run fn(g) for g in [0, G) on one host thread per device and fold the statuses (worker error texts are thread-local:
// carry them out).
template <typename Fn>
int run_per_device(int G, const int* devices, Fn fn) {
    std::vector<int> rcs(G, GPE_OK);
    std::vector<std::string> msgs(G);
    std::vector<std::thread> th;
    for (int g = 0; g < G; ++g)
        th.emplace_back([&, g] {
            bind_thread_near_device(devices[g]);
            if (cudaSetDevice(devices[g]) != cudaSuccess) rcs[g] = fail(GPE_ERR_CUDA, "cudaSetDevice(%d) failed", devices[g]);
            else rcs[g] = fn(g);
            if (rcs[g]) msgs[g] = gpe_last_error();
        });
    for (auto& t : th) t.join();
    for (int g = 0; g < G; ++g)
        if (rcs[g]) return fail(rcs[g], "device %d: %s", devices[g], msgs[g].c_str());
    return GPE_OK;
}

// Host-resident FP64 predict of one model: its share of a call of call_N points (the whole call unless `shared`
// hands out the chunks of a multi-device call).  Caller holds m->host_mu.
int model_stream(gpe_model* m, const double* testing, int64_t N, double* mu, double* var, double* deriv, double* hess,
                 const StreamPlan* shared_plan = nullptr, ChunkSource* shared = nullptr, const Relay* relay = nullptr) {
    const int64_t D = m->D;
    IoList in, out;
    in.add(testing, D);
    const int i_mu = mu ? out.add(mu, 1) : -1, i_var = var ? out.add(var, 1) : -1, i_der = deriv ? out.add(deriv, D) : -1,
              i_hes = hess ? out.add(hess, D * D) : -1;
    StreamPlan pl = shared_plan ? *shared_plan : plan_stream(in.v, in.n, out.v, out.n, N, 8, 64 * (int64_t)m->sms, 1, true);
    int rc = prepare_slots(m->slots, pl, in.v, in.n, out.v, out.n, 8);
    if (rc) return rc;
    std::atomic<int64_t> cursor{0};
    ChunkSource src = shared ? *shared : ChunkSource{&cursor, N, pl.CH};
    const int64_t call_N = src.N;   // plan choices that change the summation order follow the size of the API call
    return stream_host(m->slots, m->device, pl, src, 8, in.v, in.n, out.v, out.n,
                       [&](int64_t, int64_t n, void* const* di, void* const* dout, cudaStream_t st) {
                           auto at = [&](int i) { return i >= 0 ? (double*)dout[i] : nullptr; };
                           return predict_device(m, (const double*)di[0], n, at(i_mu), at(i_var), at(i_der), at(i_hes), 1, 1,
                                                 D, D * D, st, call_N);
                       }, relay);
}

// ---- PCA back-projection: out (R, W) = A (R, E) . basis (E, W): kernels and launcher in project.cu ----------------
constexpr int kProjCols = 128;   // columns per group of the pre-tiled basis image (project.cu)

// ---- single-precision (tcgen05 / TF32) path ------------------------------------------------------------------
uint32_t host_tf32_rna(float x) {   // round-to-nearest (ties away) to 10 mantissa bits, as cvt.rna.tf32.f32
    uint32_t u;
    memcpy(&u, &x, 4);
    if ((u & 0x7F800000u) == 0x7F800000u) return u;
    return (u + 0x1000u) & 0xFFFFE000u;
}

int ensure_tf32(gpe_model* m) {
    if (m->tf.valid) return GPE_OK;
    const int M = m->M, D = m->D;
    if (M > 1024) return fail(GPE_ERR_UNSUPPORTED, "the single-precision tensor-core path supports M <= 1024 (got %d)", M);
    int DP = -1;
    for (int dp : kTfDpList) if (dp >= D) { DP = dp; break; }
    if (DP < 0) return fail(GPE_ERR_UNSUPPORTED, "D = %d not supported by the single-precision path", D);
    const int Mp = (M + 63) / 64 * 64, nslab = (M + 31) / 32;
    // ring = true: K* slabs through a 2-deep A ring, column passes (predict_tf32_big.cuh); x3: hi + lo operands
    auto make_plan = [&](bool ring, bool x3, int pass_cols) {
        Tf32Plan t;
        t.DP = DP; t.Mp = Mp; t.nslab = nslab; t.big = ring; t.pass_cols = std::min(pass_cols, Mp);
        t.bstage_bytes = (uint32_t)(ring ? t.pass_cols : Mp) * 128u;
        uint32_t off = 0;
        t.off_bar = off; off += 128;
        t.off_tmem = off; off += 16;
        off = align_up(off, 1024);
        t.off_a = off; off += (uint32_t)(ring ? (x3 ? 4 : 2) : nslab) * kTfTN * 128u;   // A ring or the whole K* tile
        t.off_b = off; off += 2 * t.bstage_bytes;
        t.off_x = off; off += align_up((uint32_t)Mp * (DP + 1) * 4u, 16);
        t.off_out = off; off += align_up((uint32_t)kTfTN * (D + 1) * 4u, 16);
        t.off_vred = off; off += 2u * kTfTN * 4u;
        t.smem = off;
        t.valid = t.smem <= kSmemMax;
        return t;
    };
    Tf32Plan fast = (Mp <= 256) ? make_plan(false, false, Mp) : make_plan(true, false, 512);
    if (!fast.valid && Mp > 256) fast = make_plan(true, false, 256);
    // 3xTF32: M <= 256 keeps the resident-K* kernel (K*_lo lives in tensor memory), larger M the ring kernel
    Tf32Plan prec = (Mp <= 256) ? make_plan(false, false, Mp) : make_plan(true, true, 512);
    for (int pc : {256, 128, 64}) if (!prec.valid && Mp > 256) prec = make_plan(true, true, pc);
    if (!fast.valid || !prec.valid)
        return fail(GPE_ERR_UNSUPPORTED, "single-precision path does not fit shared memory for M = %d, D = %d", M, D);

    std::vector<float> xa((size_t)Mp * (DP + 1), 0.f);
    for (int j = 0; j < M; ++j) {
        for (int d = 0; d < D; ++d) xa[(size_t)j * DP + d] = (float)(m->sqrt_w[d] * m->h_inputs[(size_t)j * D + d]);
        xa[(size_t)Mp * DP + j] = (float)(m->b * m->h_invQt[j]);
    }
    CUDA_TRY(cudaMalloc((void**)&m->d_xa_f32, xa.size() * 4));
    CUDA_TRY(cudaMemcpy(m->d_xa_f32, xa.data(), xa.size() * 4, cudaMemcpyHostToDevice));
    if (!m->h_invQ.empty()) {
        // B operand: slab s holds invQ[j][32 s .. 32 s + 31] for every output column j as a [Mp][128 B] image with
        // the 16-byte chunk index XOR-ed by (j % 8): exactly what a SWIZZLE_128B K-major UMMA descriptor reads.
        // hi = rna_tf32(x); lo = rna_tf32(x - hi) for the 3 x TF32 split.
        std::vector<uint32_t> bh((size_t)nslab * Mp * 32, 0u), bl((size_t)nslab * Mp * 32, 0u);
        for (int j = 0; j < M; ++j)
            for (int i = 0; i < M; ++i) {
                const int s = i >> 5, c = (i & 31) >> 2, e = i & 3;
                const size_t at = (size_t)s * Mp * 32 + (size_t)j * 32 + (size_t)((c ^ (j & 7)) << 2) + e;
                const float x = (float)m->h_invQ[(size_t)j * M + i];
                const uint32_t hi = host_tf32_rna(x);
                float hf;
                memcpy(&hf, &hi, 4);
                bh[at] = hi;
                bl[at] = host_tf32_rna(x - hf);
            }
        CUDA_TRY(cudaMalloc((void**)&m->d_bslabs, bh.size() * 4));
        CUDA_TRY(cudaMemcpy(m->d_bslabs, bh.data(), bh.size() * 4, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMalloc((void**)&m->d_bslabs_lo, bl.size() * 4));
        CUDA_TRY(cudaMemcpy(m->d_bslabs_lo, bl.data(), bl.size() * 4, cudaMemcpyHostToDevice));
    }
    m->tf = fast;
    m->tfx = prec;
    std::vector<double>().swap(m->h_invQ);   // the FP64 host copy was only needed for this packing
    return GPE_OK;
}

int predict_device_f32(gpe_model* m, const float* testing, int64_t N, float* mu, float* var, float* deriv,
                       bool fast, cudaStream_t st) {
    if (N == 0) return GPE_OK;
    int rc = ensure_tf32(m);
    if (rc) return rc;
    if (var && !m->d_bslabs) return fail(GPE_ERR_INVALID, "variance requested but the model was created without invQ");
    const bool x3 = !fast && var != nullptr;   // without the variance both modes are plain FP32: use the lighter plan
    const Tf32Plan& t = x3 ? m->tfx : m->tf;
    const int64_t ntiles = (N + kTfTN - 1) / kTfTN;
    const int grid = (int)std::min<int64_t>(ntiles, m->sms);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (t.big) {
        Tf32BigParams p;
        memset(&p, 0, sizeof(p));
        p.testing = testing; p.N = N; p.mu = mu; p.var = var; p.deriv = deriv;
        p.ld_mu = 1; p.ld_var = 1; p.ld_deriv = m->D;
        p.xa = m->d_xa_f32; p.bslabs = m->d_bslabs; p.bslabs_lo = m->d_bslabs_lo;
        p.M = m->M; p.D = m->D; p.Mp = t.Mp; p.nslab = t.nslab; p.pass_cols = t.pass_cols; p.b = (float)m->b;
        p.off_bar = t.off_bar; p.off_a = t.off_a; p.off_b = t.off_b; p.off_x = t.off_x; p.off_out = t.off_out;
        p.off_vred = t.off_vred; p.off_tmem = t.off_tmem; p.bstage_bytes = t.bstage_bytes;
        for (int d = 0; d < 32; ++d) p.sqrt_w[d] = (float)m->sqrt_w[d];
        CUDA_TRY(launch_tf32_big(t.DP, x3, p, grid, t.smem, st));
        return GPE_OK;
    }
    Tf32Params p;
    memset(&p, 0, sizeof(p));
    p.testing = testing; p.N = N; p.mu = mu; p.var = var; p.deriv = deriv;
    p.ld_mu = 1; p.ld_var = 1; p.ld_deriv = m->D;
    p.xa = m->d_xa_f32; p.bslabs = m->d_bslabs; p.bslabs_lo = m->d_bslabs_lo;
    p.M = m->M; p.D = m->D; p.Mp = t.Mp; p.nslab = t.nslab; p.b = (float)m->b;
    p.off_bar = t.off_bar; p.off_a = t.off_a; p.off_b = t.off_b; p.off_x = t.off_x; p.off_out = t.off_out;
    p.off_vred = t.off_vred; p.off_tmem = t.off_tmem; p.bstage_bytes = t.bstage_bytes;
    for (int d = 0; d < 32; ++d) p.sqrt_w[d] = (float)m->sqrt_w[d];
    CUDA_TRY(launch_tf32(t.DP, x3, p, grid, t.smem, st));
    return GPE_OK;
}

uint64_t fnv1a(const void* data, size_t bytes, uint64_t h) {
    const uint64_t* p = (const uint64_t*)data;
    const size_t n = bytes / 8;
    for (size_t i = 0; i < n; ++i) { h ^= p[i]; h *= 1099511628211ull; }
    return h;
}

std::mutex g_wrap_mu;
gpe_model* g_wrap_model = nullptr;
uint64_t g_wrap_key = 0;

}  // namespace

namespace gpe {

int set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
int require_device(int device, int* sms) { return check_device(device, sms); }
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

}  // namespace gpe

// =================================================================================================
extern "C" {

const char* gpe_last_error(void) { return g_err; }
int gpe_version(void) { return GPE_VERSION; }
int64_t gpe_launch_count(void) { return g_launches.load(); }

// Developer aid (not part of the public header): CTA 0 of the fused kernel records clock64() at its phase
// boundaries for its first 64 tiles into `device_buf` (64 x 8 int64); pass NULL to switch tracing off.
void gpe_debug_trace(long long* device_buf) { g_trace = device_buf; }

int gpe_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int gpe_model_create(int device, int M, int D, const double* inputs, const double* expX, const double* invQt,
                     const double* invQ, gpe_model** out) {
    unsigned options = 0;
    if (const char* e = getenv("GPE_SYMMETRIC_VARIANCE")) options |= atoi(e) ? GPE_OPT_SYMMETRIC_VARIANCE : 0;
    return gpe_model_create_ex(device, M, D, inputs, expX, invQt, invQ, options, out);
}

int gpe_model_create_ex(int device, int M, int D, const double* inputs, const double* expX, const double* invQt,
                        const double* invQ, unsigned options, gpe_model** out) {
    if (!out) return fail(GPE_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (!inputs || !expX || !invQt) return fail(GPE_ERR_INVALID, "inputs, expX and invQt must be non-NULL");
    if (M < 1) return fail(GPE_ERR_INVALID, "M must be >= 1 (got %d)", M);
    if (D < 1 || D > GPE_MAX_INPUTS) return fail(GPE_ERR_INVALID, "D must be in [1, %d] (got %d)", GPE_MAX_INPUTS, D);   // 256
    int sms = 0;
    int rc = check_device(device, &sms);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(device));
    gpe_model* m = new gpe_model();
    m->device = device; m->M = M; m->D = D; m->DP = pick_dp(D); m->sms = sms;
    m->b = expX[D];
    for (int d = 0; d < 32; ++d) m->sqrt_w[d] = (d < D) ? std::sqrt(expX[d]) : 0.0;
    m->has_invQ = invQ != nullptr;
    m->symmetric = (options & GPE_OPT_SYMMETRIC_VARIANCE) != 0;
    if (D > 32) {
        // no per-D compiled kernels beyond 32 inputs: generic kernels on the K* scratch of the large-M path
        // (predict_generic.cuh); the symmetric fold does not apply (k_var_large reads the plain operand)
        m->generic = true;
        m->symmetric = false;
        m->large_Mp = (M + 63) / 64 * 64;
        m->large_kblk = m->large_Mp / 4;
        m->large_nstage = 6;
        m->large_chunk = 16 * (int64_t)m->sms * 4;
        std::vector<double> xs((size_t)M * D), al(M), sq(D);
        for (int d = 0; d < D; ++d) sq[d] = std::sqrt(expX[d]);
        for (int j = 0; j < M; ++j) {
            for (int d = 0; d < D; ++d) xs[(size_t)j * D + d] = sq[d] * inputs[(size_t)j * D + d];
            al[j] = m->b * invQt[j];
        }
        const size_t scratch = (size_t)(m->large_chunk / 16) * m->large_kblk * 64 * 8;
        cudaError_t e = cudaMalloc((void**)&m->d_gen_xs, xs.size() * 8);
        if (e == cudaSuccess) e = cudaMemcpy(m->d_gen_xs, xs.data(), xs.size() * 8, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMalloc((void**)&m->d_gen_alpha, al.size() * 8);
        if (e == cudaSuccess) e = cudaMemcpy(m->d_gen_alpha, al.data(), al.size() * 8, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMalloc((void**)&m->d_gen_sqw, sq.size() * 8);
        if (e == cudaSuccess) e = cudaMemcpy(m->d_gen_sqw, sq.data(), sq.size() * 8, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMalloc((void**)&m->d_gen_mu, (size_t)m->large_chunk * 8);
        if (e == cudaSuccess) e = cudaMalloc((void**)&m->d_kscratch, scratch);
        if (e == cudaSuccess) e = cudaMemset(m->d_kscratch, 0, scratch);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&m->scratch_free, cudaEventDisableTiming);
        if (e == cudaSuccess && invQ && M <= GPE_MAX_TRAIN) {
            const size_t Mp = (size_t)m->large_Mp;
            std::vector<double> st((size_t)m->large_kblk * Mp * 4, 0.0);
            for (int j = 0; j < M; ++j)
                for (int i = 0; i < M; ++i) st[((size_t)(i >> 2) * Mp + j) * 4 + (i & 3)] = invQ[(size_t)j * M + i];
            e = cudaMalloc((void**)&m->d_stiled, st.size() * 8);
            if (e == cudaSuccess) e = cudaMemcpy(m->d_stiled, st.data(), st.size() * 8, cudaMemcpyHostToDevice);
            m->large_valid = e == cudaSuccess;
        }
        if (e != cudaSuccess) { gpe_model_destroy(m); return fail(GPE_ERR_CUDA, "model upload failed: %s", cudaGetErrorString(e)); }
        *out = m;
        return GPE_OK;
    }
    m->h_inputs.assign(inputs, inputs + (size_t)M * D);
    m->h_invQt.assign(invQt, invQt + M);
    if (invQ && M <= 1024) m->h_invQ.assign(invQ, invQ + (size_t)M * M);
    for (int d = 0; d <= D; ++d) m->h_expx[d] = expX[d];
    m->mean = plan_mean(M, D, m->DP);
    {
        std::vector<double> xc = pack_xchunks(M, D, m->DP, m->mean.JC, m->mean.nchunks, inputs, m->sqrt_w, invQt, m->b);
        cudaError_t e = cudaMalloc((void**)&m->d_xchunks_mean, xc.size() * 8);
        if (e == cudaSuccess) e = cudaMemcpy(m->d_xchunks_mean, xc.data(), xc.size() * 8, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { gpe_model_destroy(m); return fail(GPE_ERR_CUDA, "model upload failed: %s", cudaGetErrorString(e)); }
    }
    if (invQ) {
        m->full = plan_full(M, D, m->DP);
        if (m->full.valid) {
            const FullPlan& f = m->full;
            std::vector<double> xc = pack_xchunks(M, D, m->DP, f.JC, f.nchunks, inputs, m->sqrt_w, invQt, m->b);
            // s_tiled[kb][j][c] = invQ[j][4 kb + c]
            std::vector<double> st((size_t)f.kblk * f.Mp * 4, 0.0);
            for (int j = 0; j < M; ++j)
                for (int i = 0; i < M; ++i) {
                    double v = invQ[(size_t)j * M + i];
                    if (m->symmetric)   // k^T S k = k^T T k with T_ij = S_ij + S_ji (i < j), S_jj (i == j), 0 (i > j)
                        v = (i < j) ? invQ[(size_t)j * M + i] + invQ[(size_t)i * M + j] : (i == j ? v : 0.0);
                    st[((size_t)(i >> 2) * f.Mp + j) * 4 + (i & 3)] = v;
                }
            cudaError_t e = cudaMalloc((void**)&m->d_xchunks_full, xc.size() * 8);
            if (e == cudaSuccess) e = cudaMemcpy(m->d_xchunks_full, xc.data(), xc.size() * 8, cudaMemcpyHostToDevice);
            if (e == cudaSuccess) e = cudaMalloc((void**)&m->d_stiled, st.size() * 8);
            if (e == cudaSuccess) e = cudaMemcpy(m->d_stiled, st.data(), st.size() * 8, cudaMemcpyHostToDevice);
            if (e != cudaSuccess) { gpe_model_destroy(m); return fail(GPE_ERR_CUDA, "model upload failed: %s", cudaGetErrorString(e)); }
            rc = build_hessian_operand(m, inputs, invQt);
            if (rc) { gpe_model_destroy(m); return rc; }
            // low-latency plan for small batches: a 64-point tile costs ~45 us at M = 250 even for one point
            if (f.cfg == 0 && f.Mp % 64 == 0 && getenv("GPE_NO_SMALL_PLAN") == nullptr) {
                FullPlan fs = plan_full(M, D, m->DP, f.Mp);
                if (fs.valid && fs.JC == f.JC && fs.nchunks == f.nchunks && fs.kblk == f.kblk) m->full_small = fs;
            }
        } else if (M <= GPE_MAX_TRAIN) {
            // beyond the fused kernel: s_tiled with the contraction padded to Mp (the K* scratch pads are zero)
            m->large_Mp = (M + 63) / 64 * 64;
            m->large_kblk = m->large_Mp / 4;
            m->large_nstage = 6;
            m->large_chunk = 16 * (int64_t)m->sms * 4;
            const size_t Mp = (size_t)m->large_Mp;
            std::vector<double> st((size_t)m->large_kblk * Mp * 4, 0.0);
            for (int j = 0; j < M; ++j)
                for (int i = 0; i < M; ++i) st[((size_t)(i >> 2) * Mp + j) * 4 + (i & 3)] = invQ[(size_t)j * M + i];
            const size_t scratch = (size_t)(m->large_chunk / 16) * m->large_kblk * 64 * 8;
            cudaError_t e = cudaMalloc((void**)&m->d_stiled, st.size() * 8);
            if (e == cudaSuccess) e = cudaMemcpy(m->d_stiled, st.data(), st.size() * 8, cudaMemcpyHostToDevice);
            if (e == cudaSuccess) e = cudaMalloc((void**)&m->d_kscratch, scratch);
            if (e == cudaSuccess) e = cudaMemset(m->d_kscratch, 0, scratch);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&m->scratch_free, cudaEventDisableTiming);
            if (e != cudaSuccess) { gpe_model_destroy(m); return fail(GPE_ERR_CUDA, "model upload failed: %s", cudaGetErrorString(e)); }
            m->large_valid = true;
        }
    }
    *out = m;
    return GPE_OK;
}

int gpe_model_destroy(gpe_model* m) {
    if (!m) return GPE_OK;
    cudaSetDevice(m->device);
    for (auto& s : m->slots) free_slot(s);
    if (m->d_xchunks_full) cudaFree(m->d_xchunks_full);
    if (m->d_stiled) cudaFree(m->d_stiled);
    if (m->d_ptiled) cudaFree(m->d_ptiled);
    if (m->d_kscratch) cudaFree(m->d_kscratch);
    if (m->scratch_free) cudaEventDestroy(m->scratch_free);
    if (m->d_xchunks_mean) cudaFree(m->d_xchunks_mean);
    if (m->d_gen_xs) cudaFree(m->d_gen_xs);
    if (m->d_gen_alpha) cudaFree(m->d_gen_alpha);
    if (m->d_gen_sqw) cudaFree(m->d_gen_sqw);
    if (m->d_gen_mu) cudaFree(m->d_gen_mu);
    if (m->d_xa_f32) cudaFree(m->d_xa_f32);
    if (m->d_bslabs) cudaFree(m->d_bslabs);
    if (m->d_bslabs_lo) cudaFree(m->d_bslabs_lo);
    delete m;
    return GPE_OK;
}

// Which kernel(s) a mean + variance + gradient call of N points runs on this model (bench.py reports it beside the
// roofline instead of a hard-coded name).  Returns the number of characters written.
int gpe_model_plan(gpe_model* m, int64_t N, char* buf, int len) {
    if (!m || !buf || len <= 0) return 0;
    auto full_name = [&](const FullPlan& f, char* out, int n) {
        // template arguments as instantiated in predict_full_inst.cu: <MT, NT, WR, WC, DP, MINB, KB, FULLNT, SYM, HESS>
        static const int MT[3] = {4, 4, 2}, WR[3] = {2, 1, 1}, WC[3] = {4, 8, 8}, MINB[3] = {1, 1, 1}, KB[3] = {2, 1, 1};
        const int nt_inst = f.cfg == 0 ? f.nt_act : (f.cfg == 1 ? (f.nt_act >= 5 && f.nt_act <= 7 ? f.nt_act : 8)
                                                                  : (f.nt_act >= 9 && f.nt_act <= 15 ? f.nt_act : 16));
        return snprintf(out, n, "k_predict_full<%d,%d,%d,%d,%d,%d,%d,%s,%s,false> (cfg %d: %d-point tiles, Mp=%d, %d-stage TMA ring, %u B smem)",
                        MT[f.cfg], nt_inst, WR[f.cfg], WC[f.cfg], m->DP, MINB[f.cfg], KB[f.cfg], nt_inst == f.nt_act ? "true" : "false",
                        m->symmetric ? "true" : "false", f.cfg, f.TN, f.Mp, f.nstage, f.smem);
    };
    if (m->generic)
        return snprintf(buf, len, "k_generic_kstar + k_generic_grad%s (D = %d > 32: generic kernels on the K* scratch)",
                        m->large_valid ? " + k_var_large" : "", m->D);
    if (m->has_invQ && tiny_ok(m, N))
        return snprintf(buf, len, "k_predict_tiny<%d> (one 8-CTA cluster per 16-point tile, Mp=%d)", m->DP, m->full.Mp);
    if (m->full.valid) {
        const bool small = m->full_small.valid && N <= 3 * 16 * (int64_t)m->sms;
        return full_name(small ? m->full_small : m->full, buf, len);
    }
    if (m->large_valid)
        return snprintf(buf, len, "k_predict_mean2<%d,true> + k_var_large (Mp=%d, %d k-blocks, %d-stage ring)", m->DP, m->large_Mp,
                        m->large_kblk, m->large_nstage);
    return snprintf(buf, len, "k_predict_mean2<%d,false> (no invQ: mean + gradient only)", m->DP);
}

int gpe_predict(gpe_model* m, const double* testing, int64_t N, double* mu, double* var, double* deriv, double* hess,
                unsigned flags, void* stream) {
    NvtxRange nvtx_range("gpe_predict");
    if (!m) return fail(GPE_ERR_INVALID, "model is NULL");
    if (N < 0) return fail(GPE_ERR_INVALID, "N must be >= 0");
    if (N == 0) return GPE_OK;
    if (!testing) return fail(GPE_ERR_INVALID, "testing is NULL");
    if (!(flags & GPE_WANT_MU)) mu = nullptr;
    if (!(flags & GPE_WANT_VAR)) var = nullptr;
    if (!(flags & GPE_WANT_DERIV)) deriv = nullptr;
    if (!(flags & GPE_WANT_HESS)) hess = nullptr;
    if ((flags & GPE_WANT_MU) && !mu) return fail(GPE_ERR_INVALID, "GPE_WANT_MU set but mu is NULL");
    if ((flags & GPE_WANT_VAR) && !var) return fail(GPE_ERR_INVALID, "GPE_WANT_VAR set but var is NULL");
    if ((flags & GPE_WANT_DERIV) && !deriv) return fail(GPE_ERR_INVALID, "GPE_WANT_DERIV set but deriv is NULL");
    if ((flags & GPE_WANT_HESS) && !hess) return fail(GPE_ERR_INVALID, "GPE_WANT_HESS set but hess is NULL");
    if (!mu && !var && !deriv && !hess) return fail(GPE_ERR_INVALID, "no output requested");
    CUDA_TRY(cudaSetDevice(m->device));
    if (flags & GPE_HOST_PTRS) {
        std::lock_guard<std::mutex> lock(m->host_mu);
        return model_stream(m, testing, N, mu, var, deriv, hess);
    }
    return predict_device(m, testing, N, mu, var, deriv, hess, 1, 1, m->D, (int64_t)m->D * m->D,
                          (cudaStream_t)stream);
}

int gpe_predict_f32(gpe_model* m, const float* testing, int64_t N, float* mu, float* var, float* deriv, unsigned flags,
                    void* stream) {
    if (!m) return fail(GPE_ERR_INVALID, "model is NULL");
    if (N < 0) return fail(GPE_ERR_INVALID, "N must be >= 0");
    if (N == 0) return GPE_OK;
    if (!testing) return fail(GPE_ERR_INVALID, "testing is NULL");
    if (flags & GPE_WANT_HESS) return fail(GPE_ERR_UNSUPPORTED, "the single-precision path has no Hessian output");
    if (!(flags & GPE_WANT_MU)) mu = nullptr;
    if (!(flags & GPE_WANT_VAR)) var = nullptr;
    if (!(flags & GPE_WANT_DERIV)) deriv = nullptr;
    if ((flags & GPE_WANT_MU) && !mu) return fail(GPE_ERR_INVALID, "GPE_WANT_MU set but mu is NULL");
    if ((flags & GPE_WANT_VAR) && !var) return fail(GPE_ERR_INVALID, "GPE_WANT_VAR set but var is NULL");
    if ((flags & GPE_WANT_DERIV) && !deriv) return fail(GPE_ERR_INVALID, "GPE_WANT_DERIV set but deriv is NULL");
    if (!mu && !var && !deriv) return fail(GPE_ERR_INVALID, "no output requested");
    CUDA_TRY(cudaSetDevice(m->device));
    // variance mode: 3xTF32 split unless asked otherwise -- except for M > 256, where the FP32 accumulation of the
    // long sums dominates the error anyway (1.1e-5 vs 1.5e-5 at M = 1000) and the split costs 3.6x: there the
    // single pass is the default and GPE_F32_FORCE_3X opts in
    const bool fast = (flags & GPE_F32_FAST_TF32) != 0 || (m->M > 256 && !(flags & GPE_F32_FORCE_3X));
    std::lock_guard<std::mutex> lock(m->host_mu);   // also covers the lazy packing of the FP32 operands
    if (!(flags & GPE_HOST_PTRS)) return predict_device_f32(m, testing, N, mu, var, deriv, fast, (cudaStream_t)stream);
    // host pointers: the same overlapped pipeline as the FP64 path
    const int64_t D = m->D;
    IoList in, out;
    in.add(testing, D);
    const int i_mu = mu ? out.add(mu, 1) : -1, i_var = var ? out.add(var, 1) : -1, i_der = deriv ? out.add(deriv, D) : -1;
    const StreamPlan pl = plan_stream(in.v, in.n, out.v, out.n, N, 4, 64 * (int64_t)m->sms, 1, true);
    int rc = prepare_slots(m->slots, pl, in.v, in.n, out.v, out.n, 4);
    if (rc) return rc;
    std::atomic<int64_t> cursor{0};
    return stream_host(m->slots, m->device, pl, ChunkSource{&cursor, N, pl.CH}, 4, in.v, in.n, out.v, out.n,
                       [&](int64_t, int64_t n, void* const* di, void* const* dout, cudaStream_t st) {
                           auto at = [&](int i) { return i >= 0 ? (float*)dout[i] : nullptr; };
                           return predict_device_f32(m, (const float*)di[0], n, at(i_mu), at(i_var), at(i_der), fast, st);
                       });
}

int gpe_predict_wrap(const double* expX, const double* inputs, const double* invQt, const double* invQ,
                     const double* testing, double* result, double* error, double* deriv, int Npredict, int Ntrain,
                     int Ninputs, int theta_size) {
    if (theta_size < Ninputs + 1) return fail(GPE_ERR_INVALID, "theta_size %d < Ninputs + 1", theta_size);
    if (!expX || !inputs || !invQt || !invQ || !testing || !result || !error || !deriv)
        return fail(GPE_ERR_INVALID, "NULL array argument");
    if (Npredict < 0) return fail(GPE_ERR_INVALID, "Npredict < 0");
    std::lock_guard<std::mutex> lock(g_wrap_mu);
    uint64_t key = 1469598103934665603ull ^ ((uint64_t)Ntrain << 32 | (uint32_t)Ninputs);
    key = fnv1a(expX, (size_t)(Ninputs + 1) * 8, key);
    key = fnv1a(inputs, (size_t)Ntrain * Ninputs * 8, key);
    key = fnv1a(invQt, (size_t)Ntrain * 8, key);
    key = fnv1a(invQ, (size_t)Ntrain * Ntrain * 8, key);
    if (!g_wrap_model || key != g_wrap_key) {
        if (g_wrap_model) { gpe_model_destroy(g_wrap_model); g_wrap_model = nullptr; }
        int rc = gpe_model_create(0, Ntrain, Ninputs, inputs, expX, invQt, invQ, &g_wrap_model);
        if (rc) return rc;
        g_wrap_key = key;
    }
    if (Npredict == 0) return GPE_OK;
    std::vector<double> nd((size_t)Npredict * Ninputs);
    int rc = gpe_predict(g_wrap_model, testing, Npredict, result, error, nd.data(), nullptr,
                         GPE_WANT_MU | GPE_WANT_VAR | GPE_WANT_DERIV | GPE_HOST_PTRS, nullptr);
    if (rc) return rc;
    // the legacy extension hands deriv back as (Ninputs, Npredict); its caller transposes (GaussianProcess.py:321)
    for (int n = 0; n < Npredict; ++n)
        for (int d = 0; d < Ninputs; ++d) deriv[(size_t)d * Npredict + n] = nd[(size_t)n * Ninputs + d];
    return GPE_OK;
}

}  // extern "C"

// ---- banks: E GPs sharing training inputs and test points -------------------------------------------------------
namespace {

// Device-resident bank prediction on `st`; outputs point-major: mu (N, E), var (N, E), deriv (N, E, D), hess (N, E, D, D).
int bank_predict_device(gpe_bank* b, const double* testing, int64_t N, double* mu, double* var, double* deriv, double* hess,
                        cudaStream_t stream, int64_t call_N = -1) {
    // call_N: size of the API call this launch is a chunk of -- the choice between kernels with different summation
    // orders depends on it, not on the chunk, so that one call is internally consistent (as in predict_device)
    if (call_N < 0) call_N = N;
    const int64_t E = b->E, D = b->D;
    const bool with_var = var != nullptr;
    if (b->models[0]->generic) {   // D > 32: one generic pass per emulator (predict_generic.cuh)
        for (int64_t e = 0; e < E; ++e) {
            int rc = predict_device(b->models[e], testing, N, mu ? mu + e : nullptr, var ? var + e : nullptr,
                                    deriv ? deriv + e * D : nullptr, hess ? hess + e * D * D : nullptr, E, E, E * D, E * D * D, stream, call_N);
            if (rc) return rc;
        }
        return GPE_OK;
    }
    if (with_var) {   // the variance contraction is per emulator: one fused launch each (also yields mean + gradient,
                      // and the Hessian when every emulator qualifies for the fused Hessian)
        bool fuse_hess = hess != nullptr;
        for (int64_t e = 0; e < E && fuse_hess; ++e) fuse_hess = b->models[e]->hess_fused_ok && !b->models[e]->symmetric;
        for (int64_t e = 0; e < E; ++e) {
            int rc = predict_device(b->models[e], testing, N, mu ? mu + e : nullptr, var + e, deriv ? deriv + e * D : nullptr,
                                    fuse_hess ? hess + e * D * D : nullptr, E, E, E * D, E * D * D, stream, call_N);
            if (rc) return rc;
        }
        if (fuse_hess) hess = nullptr;
    } else if (hess != nullptr && call_N >= 16384) {
        // Hessian without variance on a large batch: per-emulator fused launches (phase A + phase C) beat the
        // one-launch direct kernel when every emulator qualifies and tiles are 64 points (cfg 0)
        bool fuse_hess = true;
        for (int64_t e = 0; e < E && fuse_hess; ++e) fuse_hess = b->models[e]->hess_fused_ok && b->models[e]->full.cfg == 0;
        if (fuse_hess) {
            for (int64_t e = 0; e < E; ++e) {
                int rc = predict_device(b->models[e], testing, N, mu ? mu + e : nullptr, nullptr, deriv ? deriv + e * D : nullptr,
                                        hess + e * D * D, E, E, E * D, E * D * D, stream, call_N);
                if (rc) return rc;
            }
            return GPE_OK;
        }
    }
    // (small calls stay on the one-emulator kernel below: a thread of the group kernel does G emulators' work in sequence,
    // which only pays once its CTAs fill the machine -- one-point MultivariateEmulator.predict: 107 us against 122 us)
    if (hess == nullptr && !with_var && (mu != nullptr || deriv != nullptr) && b->gplan[deriv != nullptr].valid &&
        (call_N + kBankTN - 1) / kBankTN * b->gplan[deriv != nullptr].ngroups >= b->models[0]->sms) {
        // means (+ gradients): groups of G emulators evaluated on shared input differences (blockIdx.y = group)
        const int grad = deriv != nullptr;
        const BankMeanPlan& g = b->gplan[grad];
        gpe_model* m0 = b->models[0];
        if (g.ngroups > 65535) return fail(GPE_ERR_UNSUPPORTED, "bank size %d exceeds the grid limit", (int)E);
        BankMeanParams p;
        memset(&p, 0, sizeof(p));
        p.testing = testing; p.N = N; p.mu = mu; p.deriv = deriv;
        p.xraw = b->d_gx; p.galpha = b->d_galpha[grad]; p.gw = b->d_gw[grad];
        p.M = m0->M; p.D = m0->D; p.E = (int)E; p.JC = g.JC; p.nchunks = g.nchunks;
        p.off_x = g.off_x; p.off_a = g.off_a; p.off_w = g.off_w; p.off_ts = g.off_ts; p.smem_need = g.smem;
        const int64_t ntiles = (N + kBankTN - 1) / kBankTN;
        const int resident = grad ? 2 : 3;   // CTAs per SM (launch bounds of k_bank_mean)
        const int gx = (int)std::min<int64_t>(ntiles, std::max<int64_t>(1, (int64_t)m0->sms * resident / g.ngroups));
        CUDA_TRY(launch_bank_mean(m0->DP, g.G, grad != 0, p, dim3(gx, (unsigned)g.ngroups), g.smem, stream));
        return GPE_OK;
    }
    if (hess != nullptr || (!with_var && (mu != nullptr || deriv != nullptr))) {
        // mean / gradient / Hessian of ALL emulators in one launch (blockIdx.y = emulator)
        gpe_model* m0 = b->models[0];
        const bool do_hess = hess != nullptr;
        if (E > 65535) return fail(GPE_ERR_UNSUPPORTED, "bank size %d exceeds the grid limit", (int)E);
        MeanParams p;
        memset(&p, 0, sizeof(p));
        p.testing = testing; p.N = N;
        p.mu = with_var ? nullptr : mu;
        p.deriv = with_var ? nullptr : deriv;
        p.hess = hess;
        p.ld_mu = E; p.ld_deriv = E * D; p.ld_hess = E * D * D;
        p.eo_mu = 1; p.eo_deriv = D; p.eo_hess = D * D;
        p.bank = b->d_entries;
        p.M = m0->M; p.D = m0->D; p.JC = m0->mean.JC; p.nchunks = m0->mean.nchunks;
        p.off_xc = m0->mean.off_xc; p.off_ts = m0->mean.off_ts; p.off_out = m0->mean.off_out;
        p.smem_need = mean_extent(m0->mean, m0->D, m0->DP, do_hess);
        const int64_t ntiles = (N + kMeanTN - 1) / kMeanTN;
        const int gx = (int)std::min<int64_t>(ntiles, std::max<int64_t>(1, (int64_t)m0->sms * 8 / E));
        const size_t smem = do_hess ? m0->mean.smem_hess : m0->mean.smem;
        CUDA_TRY(launch_mean(m0->DP, do_hess, p, dim3(gx, (unsigned)E), smem, stream));
    }
    return GPE_OK;
}

// fwd (N, W) = mu (N, E) . basis, deriv_full (N, D, W) = sum_e deriv[n, e, d] basis[e, w]; banks of more than 32
// emulators run in slices of 32 that accumulate into the output (the reference has no limit on the number of PCs).
int bank_project_device(gpe_bank* b, const double* mu, const double* deriv, int64_t N, double* fwd, double* deriv_full,
                        cudaStream_t st) {
    const int E = b->E, D = b->D, W = b->W;
    auto run = [&](const double* A, int64_t R, int RD, int64_t ldn, int64_t lde, int64_t ldd, double* o) -> cudaError_t {
        for (int e0 = 0; e0 < E; e0 += 32) {
            const int Es = std::min(32, E - e0);
            g_launches.fetch_add(1);
            cudaError_t e = project_rows(A + (int64_t)e0 * lde, R, RD, ldn, lde, ldd, b->d_basis + (size_t)(e0 / 4) * b->Wp * 4, Es, W,
                                         b->Wp, o, e0 > 0, st);
            if (e != cudaSuccess) return e;
        }
        return cudaSuccess;
    };
    if (fwd) CUDA_TRY(run(mu, N, 1, E, 1, 0, fwd));
    if (deriv_full) CUDA_TRY(run(deriv, N * D, D, (int64_t)E * D, D, 1, deriv_full));
    return GPE_OK;
}

// Least-squares reduction over the emulators of a bank (SURVEY 8f-3: outputs consumed on the fly).  One warp per
// point: lanes stride over the emulators for the residuals, then lane d accumulates column d of the gradient.
__global__ void __launch_bounds__(128) k_bank_cost(const double* __restrict__ mu, const double* __restrict__ deriv,
                                                   const double* __restrict__ obs, int64_t obs_ld,
                                                   const double* __restrict__ weights, double* __restrict__ cost,
                                                   double* __restrict__ grad, int64_t n, int E, int D) {
    extern __shared__ double wr_s[];                     // [4 warps][E] weighted residuals
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    double* wr = wr_s + (size_t)w * E;
    for (int64_t pt = (int64_t)blockIdx.x * 4 + w; pt < n; pt += (int64_t)gridDim.x * 4) {
        double c = 0.0;
        for (int e = lane; e < E; e += 32) {
            const double r = mu[pt * E + e] - obs[pt * obs_ld + e];
            const double we = weights ? weights[e] : 1.0;
            wr[e] = we * r;
            c = fma(we * r, r, c);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if (lane == 0 && cost) cost[pt] = 0.5 * c;
        __syncwarp();
        if (grad != nullptr && lane < D) {
            const double* dp = deriv + pt * E * D + lane;
            double g = 0.0;
            for (int e = 0; e < E; ++e) g = fma(wr[e], dp[(size_t)e * D], g);
            grad[pt * D + lane] = g;
        }
        __syncwarp();
    }
}

int bank_cost_device(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld, const double* weights,
                     double* cost, double* grad, cudaStream_t st, int64_t call_N = -1) {
    if (call_N < 0) call_N = N;
    const int64_t E = b->E, D = b->D;
    const int64_t per_point = E * (1 + (grad ? D : 0));
    // points per chunk: whole waves of 64-point tiles, scratch bounded by 256 MB
    int64_t chunk = std::max<int64_t>(64, (((int64_t)256 << 20) / (per_point * 8)) / 64 * 64);
    chunk = std::min(chunk, (N + 63) / 64 * 64);
    std::lock_guard<std::mutex> lock(b->cost_mu);
    if (!b->cost_free) CUDA_TRY(cudaEventCreateWithFlags(&b->cost_free, cudaEventDisableTiming));
    // the scratch may still be read by a reduction enqueued on another stream
    CUDA_TRY(cudaStreamWaitEvent(st, b->cost_free, 0));
    if (b->cost_cap < (size_t)(chunk * per_point)) {
        if (b->cost_d) {
            CUDA_TRY(cudaEventSynchronize(b->cost_free));
            CUDA_TRY(cudaFree(b->cost_d));
            b->cost_d = nullptr; b->cost_cap = 0;
        }
        CUDA_TRY(cudaMalloc((void**)&b->cost_d, (size_t)(chunk * per_point) * 8));
        b->cost_cap = (size_t)(chunk * per_point);
    }
    double* d_mu = b->cost_d;
    double* d_der = grad ? b->cost_d + chunk * E : nullptr;
    const int sms = b->models[0]->sms;
    for (int64_t n0 = 0; n0 < N; n0 += chunk) {
        const int64_t n = std::min(chunk, N - n0);
        int rc = bank_predict_device(b, testing + n0 * D, n, d_mu, nullptr, d_der, nullptr, st, call_N);
        if (rc) return rc;
        const int grid = (int)std::min<int64_t>((n + 3) / 4, (int64_t)sms * 16);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        k_bank_cost<<<grid, 128, (size_t)4 * E * 8, st>>>(d_mu, d_der, obs + n0 * obs_ld, obs_ld, weights,
                                                          cost ? cost + n0 : nullptr, grad ? grad + n0 * D : nullptr, n,
                                                          (int)E, (int)D);
        CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaEventRecord(b->cost_free, st));
    return GPE_OK;
}

// Host-resident bank call through the streaming pipeline: any of the point-major bank outputs plus the back-projected
// spectra / Jacobians; the PC means / gradients a projection consumes stay on the device as chunk intermediates when
// the caller did not ask for them.  Caller holds b->host_mu.
int bank_stream(gpe_bank* b, const double* testing, int64_t N, double* mu, double* var, double* deriv, double* hess,
                double* fwd, double* deriv_full, const StreamPlan* shared_plan = nullptr, ChunkSource* shared = nullptr,
                const Relay* relay = nullptr) {
    const int64_t E = b->E, D = b->D, W = b->W;
    IoList in, out;
    in.add(testing, D);
    const int i_mu = (mu || fwd) ? out.add(mu, E) : -1;
    const int i_var = var ? out.add(var, E) : -1;
    const int i_der = (deriv || deriv_full) ? out.add(deriv, E * D) : -1;
    const int i_hes = hess ? out.add(hess, E * D * D) : -1;
    const int i_fwd = fwd ? out.add(fwd, W) : -1;
    const int i_dfl = deriv_full ? out.add(deriv_full, D * W) : -1;
    const int sms = b->models[0]->sms;
    StreamPlan pl = shared_plan ? *shared_plan : plan_stream(in.v, in.n, out.v, out.n, N, 8, 64 * (int64_t)sms, 1, true);
    int rc = prepare_slots(b->slots, pl, in.v, in.n, out.v, out.n, 8);
    if (rc) return rc;
    std::atomic<int64_t> cursor{0};
    ChunkSource src = shared ? *shared : ChunkSource{&cursor, N, pl.CH};
    return stream_host(b->slots, b->device, pl, src, 8, in.v, in.n, out.v, out.n,
                       [&](int64_t, int64_t n, void* const* di, void* const* dout, cudaStream_t st) {
                           auto at = [&](int i) { return i >= 0 ? (double*)dout[i] : nullptr; };
                           int r = bank_predict_device(b, (const double*)di[0], n, at(i_mu), at(i_var), at(i_der), at(i_hes), st, N);
                           if (r == GPE_OK && (i_fwd >= 0 || i_dfl >= 0))
                               r = bank_project_device(b, at(i_mu), at(i_der), n, at(i_fwd), at(i_dfl), st);
                           return r;
                       }, relay);
}

// Host-resident gpe_bank_cost: test points (and per-point observations) stream in, cost / gradient stream out.
int bank_cost_stream(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld, const double* weights,
                     double* cost, double* grad, const StreamPlan* shared_plan = nullptr, ChunkSource* shared = nullptr,
                     const Relay* relay = nullptr) {
    const int64_t E = b->E, D = b->D;
    if (obs_ld != 0 && obs_ld != E) return fail(GPE_ERR_INVALID, "host observations must be contiguous: obs_ld = E or 0");
    // the shared observation vector and the weights are small: one upload per call
    const size_t aux_n = (size_t)(obs_ld == 0 ? E : 0) + (weights ? E : 0);
    double *d_obs1 = nullptr, *d_w = nullptr;
    if (aux_n > 0) {
        int rc = ensure_buf((void**)&b->d_aux, &b->aux_cap, aux_n * 8, false);
        if (rc) return rc;
        double* p = b->d_aux;
        if (obs_ld == 0) { CUDA_TRY(cudaMemcpy(p, obs, (size_t)E * 8, cudaMemcpyHostToDevice)); d_obs1 = p; p += E; }
        if (weights) { CUDA_TRY(cudaMemcpy(p, weights, (size_t)E * 8, cudaMemcpyHostToDevice)); d_w = p; }
    }
    IoList in, out;
    in.add(testing, D);
    const int i_obs = obs_ld != 0 ? in.add(obs, E) : -1;
    const int i_cost = cost ? out.add(cost, 1) : -1, i_grad = grad ? out.add(grad, D) : -1;
    const int sms = b->models[0]->sms;
    StreamPlan pl = shared_plan ? *shared_plan : plan_stream(in.v, in.n, out.v, out.n, N, 8, 64 * (int64_t)sms, 1, true);
    int rc = prepare_slots(b->slots, pl, in.v, in.n, out.v, out.n, 8);
    if (rc) return rc;
    std::atomic<int64_t> cursor{0};
    ChunkSource src = shared ? *shared : ChunkSource{&cursor, N, pl.CH};
    return stream_host(b->slots, b->device, pl, src, 8, in.v, in.n, out.v, out.n,
                       [&](int64_t, int64_t n, void* const* di, void* const* dout, cudaStream_t st) {
                           return bank_cost_device(b, (const double*)di[0], n, i_obs >= 0 ? (const double*)di[i_obs] : d_obs1,
                                                   i_obs >= 0 ? E : 0, d_w, i_cost >= 0 ? (double*)dout[i_cost] : nullptr,
                                                   i_grad >= 0 ? (double*)dout[i_grad] : nullptr, st, N);
                       }, relay);
}

int bank_check_outputs(gpe_bank* b, int64_t N, const double* testing, double*& mu, double*& var, double*& deriv, double*& hess,
                       double*& fwd, double*& deriv_full, unsigned flags) {
    if (!b) return fail(GPE_ERR_INVALID, "bank is NULL");
    if (N < 0) return fail(GPE_ERR_INVALID, "N must be >= 0");
    if (N > 0 && !testing) return fail(GPE_ERR_INVALID, "testing is NULL");
    if (!(flags & GPE_WANT_MU)) mu = nullptr;
    if (!(flags & GPE_WANT_VAR)) var = nullptr;
    if (!(flags & GPE_WANT_DERIV)) deriv = nullptr;
    if (!(flags & GPE_WANT_HESS)) hess = nullptr;
    if (!(flags & GPE_WANT_FWD)) fwd = nullptr;
    if (!(flags & GPE_WANT_DERIV_FULL)) deriv_full = nullptr;
    if (((flags & GPE_WANT_MU) && !mu) || ((flags & GPE_WANT_VAR) && !var) || ((flags & GPE_WANT_DERIV) && !deriv) ||
        ((flags & GPE_WANT_HESS) && !hess) || ((flags & GPE_WANT_FWD) && !fwd) || ((flags & GPE_WANT_DERIV_FULL) && !deriv_full))
        return fail(GPE_ERR_INVALID, "an output flag is set but its array is NULL");
    if (!mu && !var && !deriv && !hess && !fwd && !deriv_full) return fail(GPE_ERR_INVALID, "no output requested");
    if (var && !b->models[0]->has_invQ) return fail(GPE_ERR_INVALID, "variance requested but the bank was created without invQ");
    if ((fwd || deriv_full) && !b->d_basis) return fail(GPE_ERR_INVALID, "bank was created without basis functions");
    return GPE_OK;
}

// Per-device PCIe rate with every device of the list copying both ways at once (what a host-resident multi-device
// call does): 16 MB pinned buffers, ~40 ms.  GB/s per direction.
std::vector<double> measure_links(const std::vector<int>& devices) {
    const int G = (int)devices.size();
    const size_t bytes = (size_t)16 << 20;
    std::vector<double> rate(G, 0.0);
    std::vector<void*> h_in(G, nullptr), h_out(G, nullptr), d_in(G, nullptr), d_out(G, nullptr);
    std::vector<cudaStream_t> s1(G, nullptr), s2(G, nullptr);
    bool ok = true;
    for (int g = 0; g < G && ok; ++g) {
        ok = cudaSetDevice(devices[g]) == cudaSuccess && cudaMallocHost(&h_in[g], bytes) == cudaSuccess &&
             cudaMallocHost(&h_out[g], bytes) == cudaSuccess && cudaMalloc(&d_in[g], bytes) == cudaSuccess &&
             cudaMalloc(&d_out[g], bytes) == cudaSuccess && cudaStreamCreateWithFlags(&s1[g], cudaStreamNonBlocking) == cudaSuccess &&
             cudaStreamCreateWithFlags(&s2[g], cudaStreamNonBlocking) == cudaSuccess;
        if (ok) memset(h_in[g], 0, bytes);
    }
    if (ok) {
        std::atomic<int> ready{0};
        std::atomic<bool> go{false};
        std::vector<std::thread> th;
        for (int g = 0; g < G; ++g)
            th.emplace_back([&, g] {
                cudaSetDevice(devices[g]);
                auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
                auto round = [&] {
                    cudaMemcpyAsync(d_in[g], h_in[g], bytes, cudaMemcpyHostToDevice, s1[g]);
                    cudaMemcpyAsync(h_out[g], d_out[g], bytes, cudaMemcpyDeviceToHost, s2[g]);
                };
                round(); cudaStreamSynchronize(s1[g]); cudaStreamSynchronize(s2[g]);     // warm
                ready++;
                while (!go.load()) {}
                const double t0 = now();
                int reps = 0;
                while (now() - t0 < 0.04) { round(); round(); cudaStreamSynchronize(s1[g]); cudaStreamSynchronize(s2[g]); reps += 2; }
                rate[g] = reps * (double)bytes / (now() - t0) / 1e9;
            });
        while (ready.load() < G) {}
        go = true;
        for (auto& t : th) t.join();
    }
    for (int g = 0; g < G; ++g) {
        if (cudaSetDevice(devices[g]) != cudaSuccess) continue;
        if (h_in[g]) cudaFreeHost(h_in[g]);
        if (h_out[g]) cudaFreeHost(h_out[g]);
        if (d_in[g]) cudaFree(d_in[g]);
        if (d_out[g]) cudaFree(d_out[g]);
        if (s1[g]) cudaStreamDestroy(s1[g]);
        if (s2[g]) cudaStreamDestroy(s2[g]);
    }
    cudaGetLastError();
    if (!ok) std::fill(rate.begin(), rate.end(), 0.0);
    return rate;
}

// Decide, once per handle, which devices send their host traffic through a partner.  GPE_MULTI_RELAY = off | auto
// (default) | force (first half of the device list relays through the second half: for tests on symmetric boxes).
// auto: a device whose measured rate is below 0.6 x the best one relays through a fast device -- on the 8-GPU boxes of
// this pool GPUs 0-3 get 6.2 GB/s per direction against 11.9 for GPUs 4-7 with all eight active, and moving ALL host
// traffic onto GPUs 4-7 lifts the aggregate from 72 to 94 GB/s per direction (profiles/r02_pcie_probe8_b.txt).
void multi_route(gpe_multi* mm) {
    std::lock_guard<std::mutex> lock(mm->route_mu);
    if (mm->routed) return;
    mm->routed = true;
    const int G = (int)mm->devices.size();
    mm->relays.assign(G, Relay());
    const char* env = getenv("GPE_MULTI_RELAY");
    const std::string mode = env ? env : "auto";
    if (G < 2 || mode == "off" || mode == "0") return;
    std::vector<int> slow, fast;
    if (mode == "force") {
        for (int g = 0; g < G; ++g) (g < G / 2 ? slow : fast).push_back(g);
    } else {
        bool distinct = true;
        for (int g = 0; g < G; ++g) for (int h = 0; h < g; ++h) distinct = distinct && mm->devices[g] != mm->devices[h];
        if (!distinct) return;
        mm->link_gbs = measure_links(mm->devices);
        const double best = *std::max_element(mm->link_gbs.begin(), mm->link_gbs.end());
        if (!(best > 0)) return;
        for (int g = 0; g < G; ++g) (mm->link_gbs[g] < 0.6 * best ? slow : fast).push_back(g);
    }
    const bool trace = getenv("GPE_PIPE_TRACE") != nullptr;
    if (trace) {
        fprintf(stderr, "[gpemu multi] link GB/s per direction (all devices copying both ways):");
        for (double v : mm->link_gbs) fprintf(stderr, " %.1f", v);
        fprintf(stderr, " | %zu slow, %zu fast\n", slow.size(), fast.size());
    }
    if (slow.empty() || fast.empty()) return;
    for (size_t i = 0; i < slow.size(); ++i) {
        const int g = slow[i], p = fast[i % fast.size()];
        const int dg = mm->devices[g], dp = mm->devices[p];
        if (dg != dp) {
            int a = 0, b = 0;
            if (cudaDeviceCanAccessPeer(&a, dg, dp) != cudaSuccess || cudaDeviceCanAccessPeer(&b, dp, dg) != cudaSuccess || !a || !b) {
                cudaGetLastError();
                continue;
            }
            cudaSetDevice(dg); cudaDeviceEnablePeerAccess(dp, 0); cudaGetLastError();   // (already enabled is fine)
            cudaSetDevice(dp); cudaDeviceEnablePeerAccess(dg, 0); cudaGetLastError();
        }
        Relay r;
        r.partner = dp;
        bool ok = cudaSetDevice(dp) == cudaSuccess;
        for (int k = 0; k < 2 && ok; ++k)
            ok = cudaStreamCreateWithFlags(&r.st[k], cudaStreamNonBlocking) == cudaSuccess &&
                 cudaEventCreateWithFlags(&r.ev_in[k], cudaEventDisableTiming) == cudaSuccess &&
                 cudaEventCreateWithFlags(&r.done[k], cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaSetDevice(dg) == cudaSuccess;
        for (int k = 0; k < 2 && ok; ++k) ok = cudaEventCreateWithFlags(&r.ev_out[k], cudaEventDisableTiming) == cudaSuccess;
        if (ok) mm->relays[g] = r;
        else cudaGetLastError();
    }
    if (trace) {
        fprintf(stderr, "[gpemu multi] relays:");
        for (int g = 0; g < G; ++g) if (mm->relays[g].partner >= 0) fprintf(stderr, " %d->%d", mm->devices[g], mm->relays[g].partner);
        fprintf(stderr, "\n");
    }
}

// The relay of pipeline g for this call (NULL: the device uses its own link), with buffers grown to the plan.
const Relay* multi_relay(gpe_multi* mm, int g, const StreamPlan& pl, const IoList& in, const IoList& out, int* rc) {
    *rc = GPE_OK;
    if (!(pl.in_direct && pl.out_direct)) return nullptr;
    Relay& r = mm->relays[g];
    if (r.partner < 0) return nullptr;
    const size_t in_b = std::max<size_t>(io_bytes(in.v, in.n, pl.CH, 8, false), 256);
    const size_t out_b = std::max<size_t>(io_bytes(out.v, out.n, pl.CH, 8, true), 256);
    if (cudaSetDevice(r.partner) != cudaSuccess) { *rc = fail(GPE_ERR_CUDA, "cudaSetDevice(%d) failed", r.partner); return nullptr; }
    for (int k = 0; k < 2 && *rc == GPE_OK; ++k) {
        *rc = ensure_buf(&r.r_in[k], &r.in_cap[k], in_b, false);
        if (*rc == GPE_OK) *rc = ensure_buf(&r.r_out[k], &r.out_cap[k], out_b, false);
    }
    cudaSetDevice(mm->devices[g]);
    return *rc == GPE_OK ? &r : nullptr;
}

void multi_free_relays(gpe_multi* mm) {
    for (size_t g = 0; g < mm->relays.size(); ++g) {
        Relay& r = mm->relays[g];
        if (r.partner < 0) continue;
        cudaSetDevice(r.partner);
        for (int k = 0; k < 2; ++k) {
            if (r.r_in[k]) cudaFree(r.r_in[k]);
            if (r.r_out[k]) cudaFree(r.r_out[k]);
            if (r.st[k]) cudaStreamDestroy(r.st[k]);
            if (r.ev_in[k]) cudaEventDestroy(r.ev_in[k]);
            if (r.done[k]) cudaEventDestroy(r.done[k]);
        }
        cudaSetDevice(mm->devices[g]);
        for (int k = 0; k < 2; ++k) if (r.ev_out[k]) cudaEventDestroy(r.ev_out[k]);
    }
    mm->relays.clear();
}

// Chunk plan of a call that G pipelines share.
StreamPlan plan_shared(const IoList& in, const IoList& out, int64_t N, int sms, int G) {
    return plan_stream(in.v, in.n, out.v, out.n, N, 8, 64 * (int64_t)sms, G, false);
}

}  // namespace

extern "C" {

int gpe_bank_create(int device, int E, int M, int D, const double* inputs, const double* expX, const double* invQt,
                    const double* invQ, const double* basis, int W, gpe_bank** out) {
    if (!out) return fail(GPE_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (E < 1) return fail(GPE_ERR_INVALID, "E must be >= 1");
    if (basis && W < 1) return fail(GPE_ERR_INVALID, "basis given but W < 1");
    gpe_bank* b = new gpe_bank();
    b->device = device; b->E = E; b->M = M; b->D = D; b->W = basis ? W : 0;
    for (int e = 0; e < E; ++e) {
        gpe_model* m = nullptr;
        int rc = gpe_model_create(device, M, D, inputs, expX + (size_t)e * (D + 1), invQt + (size_t)e * M,
                                  invQ ? invQ + (size_t)e * M * M : nullptr, &m);
        if (rc) { gpe_bank_destroy(b); return rc; }
        b->models.push_back(m);
    }
    {
        std::vector<MeanBankEntry> ent(E);
        for (int e2 = 0; e2 < E; ++e2) {
            ent[e2].xchunks = b->models[e2]->d_xchunks_mean;
            memcpy(ent[e2].sqrt_w, b->models[e2]->sqrt_w, sizeof(ent[e2].sqrt_w));
        }
        cudaError_t e = cudaMalloc((void**)&b->d_entries, sizeof(MeanBankEntry) * E);
        if (e == cudaSuccess) e = cudaMemcpy(b->d_entries, ent.data(), sizeof(MeanBankEntry) * E, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { gpe_bank_destroy(b); return fail(GPE_ERR_CUDA, "bank upload failed: %s", cudaGetErrorString(e)); }
    }
    {
        // operands of the shared-difference kernels (predict_bank_mean.cuh): [1] mean + gradient, [0] means only
        static const bool off = []{ const char* e = getenv("GPE_BANK_SHARED"); return e && !strcmp(e, "off"); }();
        const int DP = b->models[0]->DP;
        for (int grad = 0; grad < 2 && !off && !b->models[0]->generic; ++grad) {
            BankMeanPlan g = plan_bank_mean(E, M, D, DP, grad != 0);
            if (!g.valid) continue;
            const int G = g.G, GP = (G + 1) & ~1;
            std::vector<double> galpha((size_t)g.ngroups * g.nchunks * g.JC * GP, 0.0);
            std::vector<double> gw((size_t)g.ngroups * 2 * G * DP, 0.0);
            for (int e2 = 0; e2 < E; ++e2) {
                const int grp = e2 / G, el = e2 - grp * G;
                const double* ex = expX + (size_t)e2 * (D + 1);
                for (int j = 0; j < M; ++j)   // chunks are contiguous: c JC + jl = j
                    galpha[((size_t)grp * g.nchunks * g.JC + j) * GP + el] = ex[D] * invQt[(size_t)e2 * M + j];
                for (int d = 0; d < D; ++d) {
                    gw[((size_t)grp * 2 * G + el) * DP + d] = -0.5 * ex[d];
                    gw[((size_t)grp * 2 * G + G + el) * DP + d] = ex[d];
                }
            }
            cudaError_t e = cudaSuccess;
            if (!b->d_gx) {
                const int XP = x_pitch(DP);
                std::vector<double> gx((size_t)g.nchunks * g.JC * XP, 0.0);
                for (int j = 0; j < M; ++j)
                    for (int d = 0; d < D; ++d) gx[(size_t)j * XP + d] = inputs[(size_t)j * D + d];
                e = cudaMalloc((void**)&b->d_gx, gx.size() * 8);
                if (e == cudaSuccess) e = cudaMemcpy(b->d_gx, gx.data(), gx.size() * 8, cudaMemcpyHostToDevice);
            }
            if (e == cudaSuccess) e = cudaMalloc((void**)&b->d_galpha[grad], galpha.size() * 8);
            if (e == cudaSuccess) e = cudaMemcpy(b->d_galpha[grad], galpha.data(), galpha.size() * 8, cudaMemcpyHostToDevice);
            if (e == cudaSuccess) e = cudaMalloc((void**)&b->d_gw[grad], gw.size() * 8);
            if (e == cudaSuccess) e = cudaMemcpy(b->d_gw[grad], gw.data(), gw.size() * 8, cudaMemcpyHostToDevice);
            if (e != cudaSuccess) { gpe_bank_destroy(b); return fail(GPE_ERR_CUDA, "bank upload failed: %s", cudaGetErrorString(e)); }
            b->gplan[grad] = g;
        }
    }
    if (basis) {
        // k-steps of 4 emulators; the projection runs in slices of 32 emulators = 8 k-steps, and the instantiation used for
        // a slice (3, 5 or 8 k-steps) may read up to 8 k-steps from the slice's start: size the image for whole slices
        const int ks_alloc = (E + 31) / 32 * 8;
        b->Wp = (W + kProjCols - 1) / kProjCols * kProjCols;
        std::vector<double> bt((size_t)ks_alloc * b->Wp * 4, 0.0);
        for (int e2 = 0; e2 < E; ++e2)
            for (int w = 0; w < W; ++w) bt[((size_t)(e2 >> 2) * b->Wp + w) * 4 + (e2 & 3)] = basis[(size_t)e2 * W + w];
        cudaError_t e = cudaMalloc((void**)&b->d_basis, bt.size() * 8);
        if (e == cudaSuccess) e = cudaMemcpy(b->d_basis, bt.data(), bt.size() * 8, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { gpe_bank_destroy(b); return fail(GPE_ERR_CUDA, "basis upload failed: %s", cudaGetErrorString(e)); }
    }
    *out = b;
    return GPE_OK;
}

int gpe_bank_destroy(gpe_bank* b) {
    if (!b) return GPE_OK;
    cudaSetDevice(b->device);
    for (gpe_model* m : b->models) gpe_model_destroy(m);
    for (auto& s : b->slots) free_slot(s);
    if (b->d_basis) cudaFree(b->d_basis);
    if (b->d_entries) cudaFree(b->d_entries);
    if (b->d_gx) cudaFree(b->d_gx);
    for (int i = 0; i < 2; ++i) {
        if (b->d_galpha[i]) cudaFree(b->d_galpha[i]);
        if (b->d_gw[i]) cudaFree(b->d_gw[i]);
    }
    if (b->d_aux) cudaFree(b->d_aux);
    if (b->cost_d) cudaFree(b->cost_d);
    if (b->cost_free) cudaEventDestroy(b->cost_free);
    delete b;
    return GPE_OK;
}

int gpe_bank_predict_ex(gpe_bank* b, const double* testing, int64_t N, double* mu, double* var, double* deriv, double* hess,
                        double* fwd, double* deriv_full, unsigned flags, void* stream) {
    NvtxRange nvtx_range("gpe_bank_predict");
    int rc = bank_check_outputs(b, N, testing, mu, var, deriv, hess, fwd, deriv_full, flags);
    if (rc) return rc;
    if (N == 0) return GPE_OK;
    CUDA_TRY(cudaSetDevice(b->device));
    if (flags & GPE_HOST_PTRS) {
        std::lock_guard<std::mutex> lock(b->host_mu);
        return bank_stream(b, testing, N, mu, var, deriv, hess, fwd, deriv_full);
    }
    // device pointers: a projection needs the PC means / gradients materialised by the caller
    if (fwd && !mu) return fail(GPE_ERR_INVALID, "device-pointer projection: GPE_WANT_FWD needs GPE_WANT_MU (the PC means) too");
    if (deriv_full && !deriv) return fail(GPE_ERR_INVALID, "device-pointer projection: GPE_WANT_DERIV_FULL needs GPE_WANT_DERIV too");
    rc = bank_predict_device(b, testing, N, mu, var, deriv, hess, (cudaStream_t)stream);
    if (rc == GPE_OK && (fwd || deriv_full)) rc = bank_project_device(b, mu, deriv, N, fwd, deriv_full, (cudaStream_t)stream);
    return rc;
}

int gpe_bank_predict(gpe_bank* b, const double* testing, int64_t N, double* mu, double* var, double* deriv,
                     double* hess, unsigned flags, void* stream) {
    return gpe_bank_predict_ex(b, testing, N, mu, var, deriv, hess, nullptr, nullptr,
                               flags & ~(unsigned)(GPE_WANT_FWD | GPE_WANT_DERIV_FULL), stream);
}

int gpe_bank_cost(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld, const double* weights,
                  double* cost, double* grad, void* stream) {
    NvtxRange nvtx_range("gpe_bank_cost");
    if (!b) return fail(GPE_ERR_INVALID, "bank is NULL");
    if (N < 0) return fail(GPE_ERR_INVALID, "N must be >= 0");
    if (N == 0) return GPE_OK;
    if (!testing || !obs) return fail(GPE_ERR_INVALID, "testing / obs is NULL");
    if (!cost && !grad) return fail(GPE_ERR_INVALID, "no output requested");
    if (obs_ld != 0 && obs_ld < b->E) return fail(GPE_ERR_INVALID, "obs_ld must be 0 (one observation vector) or >= E");
    CUDA_TRY(cudaSetDevice(b->device));
    return bank_cost_device(b, testing, N, obs, obs_ld, weights, cost, grad, (cudaStream_t)stream);
}

int gpe_bank_cost_host(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                       const double* weights, double* cost, double* grad) {
    NvtxRange nvtx_range("gpe_bank_cost_host");
    if (!b) return fail(GPE_ERR_INVALID, "bank is NULL");
    if (N < 0) return fail(GPE_ERR_INVALID, "N must be >= 0");
    if (N == 0) return GPE_OK;
    if (!testing || !obs) return fail(GPE_ERR_INVALID, "testing / obs is NULL");
    if (!cost && !grad) return fail(GPE_ERR_INVALID, "no output requested");
    CUDA_TRY(cudaSetDevice(b->device));
    std::lock_guard<std::mutex> lock(b->host_mu);
    return bank_cost_stream(b, testing, N, obs, obs_ld, weights, cost, grad);
}

int gpe_bank_project(gpe_bank* b, const double* mu, const double* deriv, int64_t N, double* fwd, double* deriv_full,
                     void* stream) {
    if (!b) return fail(GPE_ERR_INVALID, "bank is NULL");
    if (!b->d_basis) return fail(GPE_ERR_INVALID, "bank was created without basis functions");
    if (N <= 0) return N == 0 ? GPE_OK : fail(GPE_ERR_INVALID, "N must be >= 0");
    if (fwd && !mu) return fail(GPE_ERR_INVALID, "fwd requested but mu is NULL");
    if (deriv_full && !deriv) return fail(GPE_ERR_INVALID, "deriv_full requested but deriv is NULL");
    CUDA_TRY(cudaSetDevice(b->device));
    return bank_project_device(b, mu, deriv, N, fwd, deriv_full, (cudaStream_t)stream);
}

int gpe_bank_forward(gpe_bank* b, const double* testing, int64_t N, double* fwd, double* deriv_full) {
    NvtxRange nvtx_range("gpe_bank_forward");
    if (!fwd) return fail(GPE_ERR_INVALID, "testing / fwd is NULL");
    return gpe_bank_predict_ex(b, testing, N, nullptr, nullptr, nullptr, nullptr, fwd, deriv_full,
                               GPE_WANT_FWD | (deriv_full ? GPE_WANT_DERIV_FULL : 0u) | GPE_HOST_PTRS, nullptr);
}

// ---- one call, G devices ---------------------------------------------------------------------------------------
// The model (or bank) is resident on every listed device.  A host-resident batch is cut into chunks that the devices'
// pipelines -- one host thread each -- pull from one shared cursor (SURVEY.md section 8b/8e: test points are
// independent, no steady-state exchange), so a GPU behind a slower PCIe path takes fewer chunks instead of holding the
// call back: on the 8-GPU boxes GPUs 0-3 sustain 8.0 GB/s per direction against 11.3 for GPUs 4-7 with all eight
// active (profiles/r01_pcie_8ranks.txt).
int gpe_multi_create(int n_devices, const int* devices, int M, int D, const double* inputs, const double* expX,
                     const double* invQt, const double* invQ, unsigned options, gpe_multi** out) {
    DeviceRestore restore_device;
    if (!out) return fail(GPE_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (n_devices < 1 || !devices) return fail(GPE_ERR_INVALID, "need at least one device");
    gpe_multi* mm = new gpe_multi();
    for (int i = 0; i < n_devices; ++i) {
        gpe_model* m = nullptr;
        int rc = gpe_model_create_ex(devices[i], M, D, inputs, expX, invQt, invQ, options, &m);
        if (rc) { gpe_multi_destroy(mm); return rc; }
        mm->models.push_back(m);
        mm->devices.push_back(devices[i]);
    }
    *out = mm;
    return GPE_OK;
}

int gpe_multi_bank_create(int n_devices, const int* devices, int E, int M, int D, const double* inputs, const double* expX,
                          const double* invQt, const double* invQ, const double* basis, int W, gpe_multi** out) {
    DeviceRestore restore_device;
    if (!out) return fail(GPE_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (n_devices < 1 || !devices) return fail(GPE_ERR_INVALID, "need at least one device");
    gpe_multi* mm = new gpe_multi();
    for (int i = 0; i < n_devices; ++i) {
        gpe_bank* b = nullptr;
        int rc = gpe_bank_create(devices[i], E, M, D, inputs, expX, invQt, invQ, basis, W, &b);
        if (rc) { gpe_multi_destroy(mm); return rc; }
        mm->banks.push_back(b);
        mm->devices.push_back(devices[i]);
    }
    *out = mm;
    return GPE_OK;
}

int gpe_multi_destroy(gpe_multi* mm) {
    DeviceRestore restore_device;
    if (!mm) return GPE_OK;
    multi_free_relays(mm);
    for (gpe_model* m : mm->models) gpe_model_destroy(m);
    for (gpe_bank* b : mm->banks) gpe_bank_destroy(b);
    delete mm;
    return GPE_OK;
}

int gpe_multi_predict(gpe_multi* mm, const double* testing, int64_t N, double* mu, double* var, double* deriv,
                      double* hess, unsigned flags) {
    NvtxRange nvtx_range("gpe_multi_predict");
    if (!mm || mm->models.empty()) return fail(GPE_ERR_INVALID, "handle is NULL or not a single-GP handle");
    if (N < 0) return fail(GPE_ERR_INVALID, "N must be >= 0");
    if (N == 0) return GPE_OK;
    if (!(flags & GPE_WANT_MU)) mu = nullptr;
    if (!(flags & GPE_WANT_VAR)) var = nullptr;
    if (!(flags & GPE_WANT_DERIV)) deriv = nullptr;
    if (!(flags & GPE_WANT_HESS)) hess = nullptr;
    if (((flags & GPE_WANT_MU) && !mu) || ((flags & GPE_WANT_VAR) && !var) || ((flags & GPE_WANT_DERIV) && !deriv) ||
        ((flags & GPE_WANT_HESS) && !hess) || !(mu || var || deriv || hess) || !testing)
        return fail(GPE_ERR_INVALID, "output flag set with a NULL array, or nothing requested");
    const int G = (int)mm->models.size();
    gpe_model* m0 = mm->models[0];
    const int64_t D = m0->D;
    if (G == 1 || N <= 3 * 64 * (int64_t)m0->sms) {
        // a call this small is one chunk: the first device serves it on the calling thread (no thread fan-out, and the
        // mapped-buffer path for the reference's one-point calls stays available) -- same kernels, same result
        DeviceRestore restore_device;
        CUDA_TRY(cudaSetDevice(m0->device));
        std::lock_guard<std::mutex> lock(m0->host_mu);
        return model_stream(m0, testing, N, mu, var, deriv, hess);
    }
    IoList in, out;
    in.add(testing, D);
    if (mu) out.add(mu, 1);
    if (var) out.add(var, 1);
    if (deriv) out.add(deriv, D);
    if (hess) out.add(hess, D * D);
    const StreamPlan pl = plan_shared(in, out, N, m0->sms, G);
    std::atomic<int64_t> cursor{0};
    ChunkSource src{&cursor, N, pl.CH};
    // large page-locked calls: decide (once per handle) whether some devices should send their host traffic through a
    // partner's PCIe link
    const bool relay_ok = pl.in_direct && pl.out_direct && N >= 4 * pl.CH;
    if (relay_ok) multi_route(mm);
    // the kernel plan (tile size) follows the size of the whole call, so G devices reproduce one device bit for bit
    return run_per_device(G, mm->devices.data(), [&](int g) {
        gpe_model* m = mm->models[g];
        std::lock_guard<std::mutex> lock(m->host_mu);
        int rc = GPE_OK;
        const Relay* relay = (relay_ok && mm->routed && !mm->relays.empty()) ? multi_relay(mm, g, pl, in, out, &rc) : nullptr;
        if (rc) return rc;
        return model_stream(m, testing, N, mu, var, deriv, hess, &pl, &src, relay);
    });
}

int gpe_multi_predict_device(gpe_multi* mm, const double* const* testing, const int64_t* N, double* const* mu,
                             double* const* var, double* const* deriv, double* const* hess, unsigned flags,
                             void* const* streams) {
    NvtxRange nvtx_range("gpe_multi_predict_device");
    DeviceRestore restore_device;
    if (!mm || mm->models.empty()) return fail(GPE_ERR_INVALID, "handle is NULL or not a single-GP handle");
    if (!testing || !N) return fail(GPE_ERR_INVALID, "testing / N is NULL");
    const int G = (int)mm->models.size();
    int64_t call_N = 0;
    for (int g = 0; g < G; ++g) {
        if (N[g] < 0) return fail(GPE_ERR_INVALID, "N[%d] must be >= 0", g);
        call_N += N[g];
    }
    for (int g = 0; g < G; ++g) {
        if (N[g] == 0) continue;
        gpe_model* m = mm->models[g];
        double* o_mu = (flags & GPE_WANT_MU) && mu ? mu[g] : nullptr;
        double* o_var = (flags & GPE_WANT_VAR) && var ? var[g] : nullptr;
        double* o_der = (flags & GPE_WANT_DERIV) && deriv ? deriv[g] : nullptr;
        double* o_hes = (flags & GPE_WANT_HESS) && hess ? hess[g] : nullptr;
        if (!testing[g]) return fail(GPE_ERR_INVALID, "testing[%d] is NULL", g);
        if (((flags & GPE_WANT_MU) && !o_mu) || ((flags & GPE_WANT_VAR) && !o_var) || ((flags & GPE_WANT_DERIV) && !o_der) ||
            ((flags & GPE_WANT_HESS) && !o_hes) || !(o_mu || o_var || o_der || o_hes))
            return fail(GPE_ERR_INVALID, "device %d: output flag set with a NULL array, or nothing requested", mm->devices[g]);
        CUDA_TRY(cudaSetDevice(m->device));
        int rc = predict_device(m, testing[g], N[g], o_mu, o_var, o_der, o_hes, 1, 1, m->D, (int64_t)m->D * m->D,
                                streams ? (cudaStream_t)streams[g] : nullptr, call_N);
        if (rc) return rc;
    }
    return GPE_OK;
}

int gpe_multi_bank_predict(gpe_multi* mm, const double* testing, int64_t N, double* mu, double* var, double* deriv,
                           double* hess, double* fwd, double* deriv_full, unsigned flags) {
    NvtxRange nvtx_range("gpe_multi_bank_predict");
    if (!mm || mm->banks.empty()) return fail(GPE_ERR_INVALID, "handle is NULL or not a bank handle");
    gpe_bank* b0 = mm->banks[0];
    int rc = bank_check_outputs(b0, N, testing, mu, var, deriv, hess, fwd, deriv_full, flags);
    if (rc) return rc;
    if (N == 0) return GPE_OK;
    const int G = (int)mm->banks.size();
    const int64_t E = b0->E, D = b0->D, W = b0->W;
    if (G == 1 || N <= 64 * (int64_t)b0->models[0]->sms) {   // one chunk: served by the first device on the calling thread
        DeviceRestore restore_device;
        CUDA_TRY(cudaSetDevice(b0->device));
        std::lock_guard<std::mutex> lock(b0->host_mu);
        return bank_stream(b0, testing, N, mu, var, deriv, hess, fwd, deriv_full);
    }
    IoList in, out;   // same arrays, same order as bank_stream builds them: the plan only needs widths and pinned-ness
    in.add(testing, D);
    if (mu || fwd) out.add(mu, E);
    if (var) out.add(var, E);
    if (deriv || deriv_full) out.add(deriv, E * D);
    if (hess) out.add(hess, E * D * D);
    if (fwd) out.add(fwd, W);
    if (deriv_full) out.add(deriv_full, D * W);
    const StreamPlan pl = plan_shared(in, out, N, b0->models[0]->sms, G);
    std::atomic<int64_t> cursor{0};
    ChunkSource src{&cursor, N, pl.CH};
    const bool relay_ok = pl.in_direct && pl.out_direct && N >= 4 * pl.CH;
    if (relay_ok) multi_route(mm);
    return run_per_device(G, mm->devices.data(), [&](int g) {
        gpe_bank* b = mm->banks[g];
        std::lock_guard<std::mutex> lock(b->host_mu);
        int rc = GPE_OK;
        const Relay* relay = (relay_ok && mm->routed && !mm->relays.empty()) ? multi_relay(mm, g, pl, in, out, &rc) : nullptr;
        if (rc) return rc;
        return bank_stream(b, testing, N, mu, var, deriv, hess, fwd, deriv_full, &pl, &src, relay);
    });
}

int gpe_multi_bank_cost(gpe_multi* mm, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                        const double* weights, double* cost, double* grad) {
    NvtxRange nvtx_range("gpe_multi_bank_cost");
    if (!mm || mm->banks.empty()) return fail(GPE_ERR_INVALID, "handle is NULL or not a bank handle");
    if (N < 0) return fail(GPE_ERR_INVALID, "N must be >= 0");
    if (N == 0) return GPE_OK;
    if (!testing || !obs) return fail(GPE_ERR_INVALID, "testing / obs is NULL");
    if (!cost && !grad) return fail(GPE_ERR_INVALID, "no output requested");
    gpe_bank* b0 = mm->banks[0];
    const int G = (int)mm->banks.size();
    const int64_t E = b0->E, D = b0->D;
    IoList in, out;
    in.add(testing, D);
    if (obs_ld != 0) in.add(obs, E);
    if (cost) out.add(cost, 1);
    if (grad) out.add(grad, D);
    const StreamPlan pl = plan_shared(in, out, N, b0->models[0]->sms, G);
    std::atomic<int64_t> cursor{0};
    ChunkSource src{&cursor, N, pl.CH};
    const bool relay_ok = pl.in_direct && pl.out_direct && N >= 4 * pl.CH;
    if (relay_ok) multi_route(mm);
    return run_per_device(G, mm->devices.data(), [&](int g) {
        gpe_bank* b = mm->banks[g];
        std::lock_guard<std::mutex> lock(b->host_mu);
        int rc = GPE_OK;
        const Relay* relay = (relay_ok && mm->routed && !mm->relays.empty()) ? multi_relay(mm, g, pl, in, out, &rc) : nullptr;
        if (rc) return rc;
        return bank_cost_stream(b, testing, N, obs, obs_ld, weights, cost, grad, &pl, &src, relay);
    });
}

}  // extern "C"
