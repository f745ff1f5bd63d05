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
#include "invert.h"

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
    const DpKernels* kern = nullptr;   // launchers compiled for DP (NULL: D > 32, generic kernels)
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
    cudaEvent_t aux_ready = nullptr;   // recorded after their upload, on the stream of the call's first chunk
    // gpe_bank_cost: per-chunk mu / deriv scratch, shared by every stream that reduces with this bank
    std::mutex cost_mu;
    double* cost_d = nullptr;
    size_t cost_cap = 0;
    cudaEvent_t cost_free = nullptr;
    // gpe_bank_solve: solver state and active lists (one solve at a time per bank), the active count read back per iteration
    std::mutex solve_mu;
    void* solve_d = nullptr;
    size_t solve_cap = 0;
    int* solve_count = nullptr;        // page-locked
    cudaEvent_t solve_ev = nullptr;
    // gpe_bank_search: candidate table and per-pixel scratch (one search at a time per bank), handed between streams
    // through search_free
    std::mutex search_mu;
    void* search_d = nullptr;
    size_t search_cap = 0;
    cudaEvent_t search_free = nullptr;
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

// cudaMalloc + copy of a host image.
template <typename T>
cudaError_t upload(T** d, const std::vector<T>& h) {
    const cudaError_t e = cudaMalloc((void**)d, h.size() * sizeof(T));
    return e == cudaSuccess ? cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice) : e;
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

cudaError_t build_hessian_operand(gpe_model* m, const double* inputs, const double* invQt) {
    const FullPlan& f = m->full;
    const int M = m->M, D = m->D;
    memset(m->centre, 0, sizeof(m->centre));
    m->hess_fused_ok = false;
    if (getenv("GPE_HESS_DIRECT") != nullptr) return cudaSuccess;   // dev aid: always use the direct Hessian kernels
    if (!f.valid || f.kbh < 1 || f.NC > M || f.NC > f.Mp) return cudaSuccess;
    double r2max = 0.0;
    for (int d = 0; d < D; ++d) {
        double lo = inputs[d], hi = inputs[d];
        for (int j = 1; j < M; ++j) { lo = std::min(lo, inputs[(size_t)j * D + d]); hi = std::max(hi, inputs[(size_t)j * D + d]); }
        m->centre[d] = m->sqrt_w[d] * 0.5 * (lo + hi);
        const double r = m->sqrt_w[d] * 0.5 * (hi - lo);
        r2max = std::max(r2max, r * r);
    }
    if (!(r2max <= kHessFusedMaxR2)) return cudaSuccess;
    std::vector<double> pt((size_t)f.kblk * f.NC * 4, 0.0);
    std::vector<double> xp(D);
    for (int j = 0; j < M; ++j) {
        for (int d = 0; d < D; ++d) xp[d] = m->sqrt_w[d] * inputs[(size_t)j * D + d] - m->centre[d];
        const double ba = m->b * invQt[j];
        int col = 0;
        for (int d = 0; d < D; ++d)
            for (int e = d; e < D; ++e, ++col) pt[((size_t)(j >> 2) * f.NC + col) * 4 + (j & 3)] = ba * xp[d] * xp[e];
    }
    const cudaError_t e = upload(&m->d_ptiled, pt);
    m->hess_fused_ok = e == cudaSuccess;
    return e;
}

// K* scratch of the two-launch variance path (1024 < M <= GPE_MAX_TRAIN) and of the generic kernels (D > 32), and with
// invQ the s_tiled image with the contraction padded to Mp (the scratch pads are zero): d_stiled then has Mp / 4 k-blocks.
cudaError_t setup_large(gpe_model* m, const double* invQ) {
    const int M = m->M;
    m->large_Mp = (M + 63) / 64 * 64;
    m->large_kblk = m->large_Mp / 4;
    m->large_nstage = 6;
    m->large_chunk = 16 * (int64_t)m->sms * 4;
    const size_t scratch = (size_t)(m->large_chunk / 16) * m->large_kblk * 64 * 8;
    cudaError_t e = cudaMalloc((void**)&m->d_kscratch, scratch);
    if (e == cudaSuccess) e = cudaMemset(m->d_kscratch, 0, scratch);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&m->scratch_free, cudaEventDisableTiming);
    if (e != cudaSuccess || !invQ || M > GPE_MAX_TRAIN) return e;
    const size_t Mp = (size_t)m->large_Mp;
    std::vector<double> st((size_t)m->large_kblk * Mp * 4, 0.0);
    for (int j = 0; j < M; ++j)
        for (int i = 0; i < M; ++i) st[((size_t)(i >> 2) * Mp + j) * 4 + (i & 3)] = invQ[(size_t)j * M + i];
    e = upload(&m->d_stiled, st);
    m->large_valid = e == cudaSuccess;
    return e;
}

// k_var_large over n points whose K* is in the model's scratch (1024 < M <= GPE_MAX_TRAIN, and D > 32).
cudaError_t var_large(const gpe_model* m, double* var, int64_t ld_var, int64_t n, cudaStream_t st) {
    VarLargeParams v;
    memset(&v, 0, sizeof(v));
    v.kstar = m->d_kscratch; v.s_tiled = m->d_stiled; v.var = var; v.ld_var = ld_var; v.N = n;
    v.Mp = m->large_Mp; v.kblk = m->large_kblk; v.npass = (m->large_Mp + kVlPass - 1) / kVlPass;
    v.nstage = m->large_nstage; v.b = m->b;
    const size_t smem = 128 + kVlWarps * kVlTN * 8 + (size_t)v.nstage * kVlStageBytes;
    return launch_var_large(v, (int)std::min<int64_t>((n + kVlTN - 1) / kVlTN, m->sms), smem, st);
}

// D > 32 (predict_generic.cuh): K* of a sub-batch into the model's scratch, then gradient / variance / Hessian from it.
int predict_generic(gpe_model* m, const double* testing, int64_t N, double* mu, double* var, double* deriv, double* hess,
                    int64_t ld_mu, int64_t ld_var, int64_t ld_deriv, int64_t ld_hess, cudaStream_t st) {
    if (var != nullptr && !m->has_invQ) return fail(GPE_ERR_INVALID, "variance requested but the model was created without invQ");
    if (var != nullptr && !m->large_valid)
        return fail(GPE_ERR_UNSUPPORTED, "variance contraction supports M <= %d (got M = %d)", GPE_MAX_TRAIN, m->M);
    const int D = m->D;
    const size_t smem_k = ((size_t)(kGenTN + kGenJC) * (D + 1) + 128) * 8;
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
        CUDA_TRY(launch_kernel(k_generic_kstar, (unsigned)std::min<int64_t>(tiles, (int64_t)m->sms * 4), kGenThreads, smem_k, st, p));
        if (deriv != nullptr)
            CUDA_TRY(launch_kernel(k_generic_grad, dim3((unsigned)std::min<int64_t>(tiles, (int64_t)m->sms * 8), (unsigned)std::min((D + 15) / 16, 16)),
                                   kGenThreads, 0, st, p));
        if (var != nullptr) CUDA_TRY(var_large(m, var + n0 * ld_var, ld_var, n, st));
        if (hess != nullptr) CUDA_TRY(launch_kernel(k_generic_hess, (unsigned)std::min<int64_t>(n, (int64_t)m->sms * 8), kGenThreads, 0, st, p));
    }
    CUDA_TRY(cudaEventRecord(m->scratch_free, st));
    return GPE_OK;
}

// Which kernels a call of call_N points runs on a model: predict_device follows it, gpe_model_plan reports it.
enum class Path { generic, large, tiny, fused, mean };
struct CallPlan {
    Path path;                        // what computes a variance (mean: the model has no variance path)
    const FullPlan* full = nullptr;   // plan of a fused launch: the main one, or 16-point tiles for a small call
    bool fuse_hess = false;           // a requested Hessian rides on the fused launch
};

CallPlan plan_call(const gpe_model* m, int64_t call_N, bool var, bool hess) {
    CallPlan c;
    if (m->generic) { c.path = Path::generic; return c; }
    // The cluster path for a mean + variance + gradient call (predict_tiny.cuh): the fused plan's resident training
    // chunk, a compiled DP, and few enough points (GPE_TINY_MAX overrides the threshold, GPE_NO_TINY disables).
    static const bool no_tiny = getenv("GPE_NO_TINY") != nullptr;
    static const int64_t env_max = getenv("GPE_TINY_MAX") ? atoll(getenv("GPE_TINY_MAX")) : -1;
    // two clusters per 8 SMs: measured at M = 250 (tools/tiny_threshold_probe.py, synchronous device calls) the cluster path
    // takes 37.9 us against 49.3 us at 500 points and draws level with the 16-point plan at 1000
    const int64_t tiny_max = env_max >= 0 ? env_max : kTinyTN * (int64_t)(2 * m->sms / kTinyCluster);
    const FullPlan& f = m->full;
    const bool tiny = m->has_invQ && !no_tiny && f.valid && f.cfg == 0 && f.nchunks == 1 && m->DP <= 16 && call_N <= tiny_max;
    c.path = tiny ? Path::tiny : f.valid ? Path::fused : m->large_valid ? Path::large : Path::mean;
    // the Hessian rides on the fused kernel when the model qualifies (build_hessian_operand); without a variance
    // request that only pays for the 64-point tiles of cfg 0 (measured: 4.6e8 vs 3.6e8 points/s at M = 250, but
    // 0.98e8 vs 1.10e8 at M = 1000), so larger M keeps the direct kernel for Hessian-only calls
    // (the HESS variants are built on the plain variance operand: with a symmetric-folded model the Hessian only rides
    // along when no variance is requested -- phase B is then skipped and the fold does not matter)
    // (calls small enough for the cluster path take the variance from it whatever else is requested, and the Hessian
    // from the direct kernel: every output of a call of a given size comes from the same kernel for any combination of flags)
    c.fuse_hess = hess && m->hess_fused_ok && !tiny && (var ? !m->symmetric : f.cfg == 0);
    // up to three waves of 16-point tiles finish sooner than one wave of 64-point tiles
    const bool small = m->full_small.valid && !c.fuse_hess && call_N <= 3 * 16 * (int64_t)m->sms;
    c.full = small ? &m->full_small : &m->full;
    return c;
}

// Launch the kernels for device-resident data on `st`.  Output strides allow bank (point-major) layouts.
int predict_device(gpe_model* m, const double* testing, int64_t N, double* mu, double* var, double* deriv,
                   double* hess, int64_t ld_mu, int64_t ld_var, int64_t ld_deriv, int64_t ld_hess,
                   cudaStream_t st, int64_t call_N = -1) {
    // call_N: size of the API call this launch is a chunk of (the host pipeline); plan choices that change the
    // summation order depend on it, not on the chunk, so that one call is internally consistent
    if (call_N < 0) call_N = N;
    if (N == 0) return GPE_OK;
    const CallPlan c = plan_call(m, call_N, var != nullptr, hess != nullptr);
    if (c.path == Path::generic) return predict_generic(m, testing, N, mu, var, deriv, hess, ld_mu, ld_var, ld_deriv, ld_hess, st);
    bool mean_done = false;
    static const bool force_full = getenv("GPE_FORCE_FULL") != nullptr;  // dev aid: time phase A alone
    if (var != nullptr && c.path == Path::large) {
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
            CUDA_TRY(m->kern->mean(false, p, dim3((unsigned)std::min<int64_t>(mtiles, (int64_t)m->sms * 12)), m->mean.smem, st));
            CUDA_TRY(var_large(m, var + n0 * ld_var, ld_var, n, st));
        }
        CUDA_TRY(cudaEventRecord(m->scratch_free, st));
        mean_done = true;
        var = nullptr;
    }
    // A handful of points (up to two clusters per 8 SMs): the latency path, one 8-CTA cluster per 16-point tile
    // (predict_tiny.cuh).  Needs the fused plan's resident training chunk; a Hessian request goes the usual way.
    if (var != nullptr && c.path == Path::tiny) {
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
        CUDA_TRY(m->kern->tiny(p, grid, smem, st));
        mean_done = true;
        var = nullptr;
    }
    if (var != nullptr || c.fuse_hess || (force_full && m->full.valid)) {
        if (var != nullptr && !m->has_invQ) return fail(GPE_ERR_INVALID, "variance requested but the model was created without invQ");
        if (!m->full.valid)
            return fail(GPE_ERR_UNSUPPORTED, "variance contraction supports M <= %d (got M = %d)", GPE_MAX_TRAIN, m->M);
        const FullPlan& f = *c.full;
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
        if (c.fuse_hess) {
            p.hess = hess; p.ld_hess = ld_hess; p.p_tiled = m->d_ptiled; p.kbh = f.kbh; p.nit_h = f.nit_h; p.off_hts = f.off_hts;
            memcpy(p.centre, m->centre, sizeof(p.centre));
            hess = nullptr;   // done by this launch
        }
        const int64_t ntiles = (N + f.TN - 1) / f.TN;
        const int grid = (int)std::min<int64_t>(ntiles, (int64_t)m->sms * f.ctas_per_sm);
        CUDA_TRY(m->kern->full(f.cfg, p, grid, f.smem, st));
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
        CUDA_TRY(m->kern->mean(do_hess, p, dim3(grid), smem, st));
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

// Request check of every entry point.  outs are the entry point's output arrays in GPE_WANT_* bit order (mu, var,
// deriv, hess, fwd, deriv_full), as many as it has: an array whose flag is clear is dropped; a set flag with a NULL
// array, or a call that asks for nothing, is an error.
template <typename... T>
int take_outputs(unsigned flags, T*&... outs) {
    unsigned bit = GPE_WANT_MU;
    bool missing = false, any = false;
    auto take = [&](auto*& o) {
        if (!(flags & bit)) o = nullptr;
        else if (!o) missing = true;
        any = any || o != nullptr;
        bit <<= 1;
    };
    (take(outs), ...);
    if (missing) return fail(GPE_ERR_INVALID, "an output flag is set but its array is NULL");
    if (!any) return fail(GPE_ERR_INVALID, "no output requested");
    return GPE_OK;
}

// The streamed arrays of one host-resident call, in the order its chunk launch reads them: idx[k] is the chunk array
// of the call kind's k-th array (-1: not streamed).
struct CallIo {
    IoList in, out;
    int idx[6] = {-1, -1, -1, -1, -1, -1};
    template <typename T>
    T* at(void* const* chunk, int k) const { return idx[k] >= 0 ? (T*)chunk[idx[k]] : nullptr; }
};

// Single GP: testing in; mu, var, deriv, hess out (idx 0-3).
CallIo model_io(int64_t D, const void* testing, const void* mu, const void* var, const void* deriv, const void* hess) {
    CallIo io;
    io.in.add(testing, D);
    io.idx[0] = mu ? io.out.add(mu, 1) : -1;
    io.idx[1] = var ? io.out.add(var, 1) : -1;
    io.idx[2] = deriv ? io.out.add(deriv, D) : -1;
    io.idx[3] = hess ? io.out.add(hess, D * D) : -1;
    return io;
}

// The part of a multi-device call that one pipeline runs: the call's shared chunk plan and cursor, the device's relay.
struct SharedCall {
    const StreamPlan* plan;
    ChunkSource* src;
    const Relay* relay;
};

// Chunk plan of a call of N points: for one pipeline of its own (shared_by = 0: the mapped-buffer path is open to tiny
// calls), or shared by that many pipelines pulling from one cursor.
StreamPlan stream_plan(const CallIo& io, int64_t N, size_t ES, int sms, int shared_by = 0) {
    return plan_stream(io.in.v, io.in.n, io.out.v, io.out.n, N, ES, 64 * (int64_t)sms, std::max(shared_by, 1), shared_by == 0);
}

// Run a host-resident call of N points through an owner's slots (caller holds the owner's host_mu): with a plan and a
// cursor of its own, or with `shared` its share of a multi-device call.  launch(n0, n, d_ins, d_outs, stream) enqueues
// the kernels of one chunk (host_stream.h).
template <typename Launch>
int stream_call(Slot* slots, int device, int sms, const CallIo& io, int64_t N, size_t ES, const SharedCall* shared,
                Launch launch) {
    const StreamPlan pl = shared ? *shared->plan : stream_plan(io, N, ES, sms);
    int rc = prepare_slots(slots, pl, io.in.v, io.in.n, io.out.v, io.out.n, ES);
    if (rc) return rc;
    std::atomic<int64_t> cursor{0};
    const ChunkSource src = shared ? *shared->src : ChunkSource{&cursor, N, pl.CH};
    return stream_host(slots, device, pl, src, ES, io.in.v, io.in.n, io.out.v, io.out.n, launch, shared ? shared->relay : nullptr);
}

// Host-resident FP64 predict of one model.  Plan choices that change the summation order follow the size N of the API
// call, not of a chunk.
int model_stream(gpe_model* m, int64_t N, const CallIo& io, const SharedCall* shared = nullptr) {
    const int64_t D = m->D;
    return stream_call(m->slots, m->device, m->sms, io, N, 8, shared,
                       [&](int64_t, int64_t n, void* const* di, void* const* dout, cudaStream_t st) {
                           return predict_device(m, (const double*)di[0], n, io.at<double>(dout, 0), io.at<double>(dout, 1),
                                                 io.at<double>(dout, 2), io.at<double>(dout, 3), 1, 1, D, D * D, st, N);
                       });
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
    CUDA_TRY(upload(&m->d_xa_f32, xa));
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
        CUDA_TRY(upload(&m->d_bslabs, bh));
        CUDA_TRY(upload(&m->d_bslabs_lo, bl));
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
    m->device = device; m->M = M; m->D = D; m->sms = sms;
    m->kern = dp_kernels(D);
    m->DP = m->kern ? m->kern->DP : -1;
    m->b = expX[D];
    for (int d = 0; d < 32; ++d) m->sqrt_w[d] = (d < D) ? std::sqrt(expX[d]) : 0.0;
    m->has_invQ = invQ != nullptr;
    m->symmetric = (options & GPE_OPT_SYMMETRIC_VARIANCE) != 0;
    if (D > 32) {
        // no per-D compiled kernels beyond 32 inputs: generic kernels on the K* scratch of the large-M path
        // (predict_generic.cuh); the symmetric fold does not apply (k_var_large reads the plain operand)
        m->generic = true;
        m->symmetric = false;
        std::vector<double> xs((size_t)M * D), al(M), sq(D);
        for (int d = 0; d < D; ++d) sq[d] = std::sqrt(expX[d]);
        for (int j = 0; j < M; ++j) {
            for (int d = 0; d < D; ++d) xs[(size_t)j * D + d] = sq[d] * inputs[(size_t)j * D + d];
            al[j] = m->b * invQt[j];
        }
        cudaError_t e = setup_large(m, invQ);
        if (e == cudaSuccess) e = upload(&m->d_gen_xs, xs);
        if (e == cudaSuccess) e = upload(&m->d_gen_alpha, al);
        if (e == cudaSuccess) e = upload(&m->d_gen_sqw, sq);
        if (e == cudaSuccess) e = cudaMalloc((void**)&m->d_gen_mu, (size_t)m->large_chunk * 8);
        if (e != cudaSuccess) { gpe_model_destroy(m); return fail(GPE_ERR_CUDA, "model upload failed: %s", cudaGetErrorString(e)); }
        *out = m;
        return GPE_OK;
    }
    m->h_inputs.assign(inputs, inputs + (size_t)M * D);
    m->h_invQt.assign(invQt, invQt + M);
    if (invQ && M <= 1024) m->h_invQ.assign(invQ, invQ + (size_t)M * M);
    for (int d = 0; d <= D; ++d) m->h_expx[d] = expX[d];
    m->mean = plan_mean(M, D, m->DP);
    cudaError_t e = upload(&m->d_xchunks_mean, pack_xchunks(M, D, m->DP, m->mean.JC, m->mean.nchunks, inputs, m->sqrt_w, invQt, m->b));
    if (e == cudaSuccess && invQ) {
        m->full = plan_full(M, D, m->DP);
        if (m->full.valid) {
            const FullPlan& f = m->full;
            // s_tiled[kb][j][c] = invQ[j][4 kb + c]
            std::vector<double> st((size_t)f.kblk * f.Mp * 4, 0.0);
            for (int j = 0; j < M; ++j)
                for (int i = 0; i < M; ++i) {
                    double v = invQ[(size_t)j * M + i];
                    if (m->symmetric)   // k^T S k = k^T T k with T_ij = S_ij + S_ji (i < j), S_jj (i == j), 0 (i > j)
                        v = (i < j) ? invQ[(size_t)j * M + i] + invQ[(size_t)i * M + j] : (i == j ? v : 0.0);
                    st[((size_t)(i >> 2) * f.Mp + j) * 4 + (i & 3)] = v;
                }
            e = upload(&m->d_xchunks_full, pack_xchunks(M, D, m->DP, f.JC, f.nchunks, inputs, m->sqrt_w, invQt, m->b));
            if (e == cudaSuccess) e = upload(&m->d_stiled, st);
            if (e == cudaSuccess) e = build_hessian_operand(m, inputs, invQt);
            // low-latency plan for small batches: a 64-point tile costs ~45 us at M = 250 even for one point
            if (f.cfg == 0 && f.Mp % 64 == 0 && getenv("GPE_NO_SMALL_PLAN") == nullptr) {
                FullPlan fs = plan_full(M, D, m->DP, f.Mp);
                if (fs.valid && fs.JC == f.JC && fs.nchunks == f.nchunks && fs.kblk == f.kblk) m->full_small = fs;
            }
        } else if (M <= GPE_MAX_TRAIN) {
            e = setup_large(m, invQ);   // beyond the fused kernel: the two-launch variance path
        }
    }
    if (e != cudaSuccess) { gpe_model_destroy(m); return fail(GPE_ERR_CUDA, "model upload failed: %s", cudaGetErrorString(e)); }
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
    const CallPlan c = plan_call(m, N, true, false);
    switch (c.path) {
        case Path::generic:
            return snprintf(buf, len, "k_generic_kstar + k_generic_grad%s (D = %d > 32: generic kernels on the K* scratch)",
                            m->large_valid ? " + k_var_large" : "", m->D);
        case Path::tiny:
            return snprintf(buf, len, "k_predict_tiny<%d> (one 8-CTA cluster per 16-point tile, Mp=%d)", m->DP, m->full.Mp);
        case Path::fused: {
            const FullPlan& f = *c.full;
            const int n = std::min(m->kern->full_name(f.cfg, f.nt_act, m->symmetric, buf, len), len - 1);
            return n + snprintf(buf + n, len - n, " (cfg %d: %d-point tiles, Mp=%d, %d-stage TMA ring, %u B smem, JC=%d, nchunks=%d)",
                                f.cfg, f.TN, f.Mp, f.nstage, f.smem, f.JC, f.nchunks);
        }
        case Path::large:
            return snprintf(buf, len, "k_predict_mean2<%d,true> + k_var_large (Mp=%d, %d k-blocks, %d-stage ring)", m->DP,
                            m->large_Mp, m->large_kblk, m->large_nstage);
        case Path::mean: break;
    }
    return snprintf(buf, len, "%s<%d,false> (no invQ: mean + gradient only)", m->kern->mean_name(), m->DP);
}

int gpe_predict(gpe_model* m, const double* testing, int64_t N, double* mu, double* var, double* deriv, double* hess,
                unsigned flags, void* stream) {
    NvtxRange nvtx_range("gpe_predict");
    if (!m) return fail(GPE_ERR_INVALID, "model is NULL");
    if (N < 0) return fail(GPE_ERR_INVALID, "N must be >= 0");
    if (N == 0) return GPE_OK;
    if (!testing) return fail(GPE_ERR_INVALID, "testing is NULL");
    int rc = take_outputs(flags, mu, var, deriv, hess);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(m->device));
    if (flags & GPE_HOST_PTRS) {
        std::lock_guard<std::mutex> lock(m->host_mu);
        return model_stream(m, N, model_io(m->D, testing, mu, var, deriv, hess));
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
    int rc = take_outputs(flags, mu, var, deriv);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(m->device));
    // variance mode: 3xTF32 split unless asked otherwise -- except for M > 256, where the FP32 accumulation of the
    // long sums dominates the error anyway (1.1e-5 vs 1.5e-5 at M = 1000) and the split costs 3.6x: there the
    // single pass is the default and GPE_F32_FORCE_3X opts in
    const bool fast = (flags & GPE_F32_FAST_TF32) != 0 || (m->M > 256 && !(flags & GPE_F32_FORCE_3X));
    std::lock_guard<std::mutex> lock(m->host_mu);   // also covers the lazy packing of the FP32 operands
    if (!(flags & GPE_HOST_PTRS)) return predict_device_f32(m, testing, N, mu, var, deriv, fast, (cudaStream_t)stream);
    // host pointers: the same overlapped pipeline as the FP64 path
    const CallIo io = model_io(m->D, testing, mu, var, deriv, nullptr);
    return stream_call(m->slots, m->device, m->sms, io, N, 4, nullptr,
                       [&](int64_t, int64_t n, void* const* di, void* const* dout, cudaStream_t st) {
                           return predict_device_f32(m, (const float*)di[0], n, io.at<float>(dout, 0), io.at<float>(dout, 1),
                                                     io.at<float>(dout, 2), fast, st);
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
        CUDA_TRY(m0->kern->bank_mean(g.G, grad != 0, p, dim3(gx, (unsigned)g.ngroups), g.smem, stream));
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
        CUDA_TRY(m0->kern->mean(do_hess, p, dim3(gx, (unsigned)E), smem, stream));
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
// PW: per-point weights, row pt at weights + pt * w_ld (DESIGN 4.6f); otherwise one shared row.
template <bool PW>
__global__ void __launch_bounds__(128) k_bank_cost(const double* __restrict__ mu, const double* __restrict__ deriv,
                                                   const double* __restrict__ obs, int64_t obs_ld,
                                                   const double* __restrict__ weights, double* __restrict__ cost,
                                                   double* __restrict__ grad, int64_t n, int E, int D, int64_t w_ld) {
    extern __shared__ double wr_s[];                     // [4 warps][E] weighted residuals
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    double* wr = wr_s + (size_t)w * E;
    for (int64_t pt = (int64_t)blockIdx.x * 4 + w; pt < n; pt += (int64_t)gridDim.x * 4) {
        double c = 0.0;
        for (int e = lane; e < E; e += 32) {
            const double r = mu[pt * E + e] - obs[pt * obs_ld + e];
            const double we = weights ? weights[(PW ? pt * w_ld : 0) + e] : 1.0;
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

// Exact Hessian of a bank cost, per point (DESIGN 4.6c), from the chunk scratch of bank_cost_walk:
//   hess_n = sum_e c_ne H_ne + G_n^T A G_n,   G_n = deriv (E, D), H_ne = hs (E, D, D)
//   band cost (s == NULL):     c = w o (mu - obs), formed here; A = diag(w) (C == NULL)
//   forward cost (s != NULL):  c = s (n, E) from k_forward_cost;  A = C (E, E) from k_forward_cost_curv
// A CTA takes P points at a time: their c (and, with C, T = C G_n) go to shared memory, then one thread per point and
// upper-triangle entry i <= j sums over e in ascending order and writes (i, j) and (j, i): hess_n == hess_n^T bit for bit.
// PW (DESIGN 4.6f): per-point weights w_n at weights + pt * w_ld, and one C_n (E, E) per point at C + pt E^2.
template <bool PW>
__global__ void __launch_bounds__(256) k_cost_hess(const double* __restrict__ mu, const double* __restrict__ obs, int64_t obs_ld,
                                                   const double* __restrict__ weights, const double* __restrict__ s,
                                                   const double* __restrict__ C, const double* __restrict__ deriv,
                                                   const double* __restrict__ hs, int64_t n, int E, int D, int P,
                                                   double* __restrict__ hess, int64_t w_ld) {
    extern __shared__ double ch_s[];                     // [P][E] c, then (C) [P][E][D] T
    double* cs = ch_s;
    double* T = ch_s + (size_t)P * E;
    const int tid = threadIdx.x, nt = D * (D + 1) / 2;
    const int64_t ED = (int64_t)E * D, EDD = ED * D;
    for (int64_t p0 = (int64_t)blockIdx.x * P; p0 < n; p0 += (int64_t)gridDim.x * P) {
        const int np = n - p0 < P ? (int)(n - p0) : P;
        for (int k = tid; k < np * E; k += blockDim.x) {
            const int pl = k / E, e = k - pl * E;
            const int64_t pt = p0 + pl;
            cs[k] = s ? s[pt * E + e] : (weights ? weights[(PW ? pt * w_ld : 0) + e] : 1.0) * (mu[pt * E + e] - obs[pt * obs_ld + e]);
        }
        if (C) {
            for (int64_t k = tid; k < np * ED; k += blockDim.x) {
                const int pl = (int)(k / ED), e = (int)((k - pl * ED) / D), d = (int)(k - pl * ED - (int64_t)e * D);
                const double* g = deriv + (p0 + pl) * ED + d;
                const double* Cn = PW ? C + (p0 + pl) * E * E : C;
                double v = 0.0;
                for (int f = 0; f < E; ++f) v = fma(Cn[(int64_t)e * E + f], g[(int64_t)f * D], v);
                T[k] = v;
            }
        }
        __syncthreads();
        for (int k = tid; k < np * nt; k += blockDim.x) {
            const int pl = k / nt;
            int q = k - pl * nt, i = 0;
            while (q >= D - i) { q -= D - i; ++i; }
            const int j = i + q;
            const int64_t pt = p0 + pl;
            const double* g = deriv + pt * ED;
            const double* h = hs + pt * EDD + i * D + j;
            const double* c = cs + (size_t)pl * E;
            double a = 0.0, gn = 0.0;
            for (int e = 0; e < E; ++e) a = fma(c[e], h[(int64_t)e * D * D], a);
            if (C) {
                const double* t = T + (size_t)pl * ED + j;
                for (int e = 0; e < E; ++e) gn = fma(g[(int64_t)e * D + i], t[(int64_t)e * D], gn);
            } else {
                const double* wn = PW && weights ? weights + pt * w_ld : weights;
                for (int e = 0; e < E; ++e) gn = fma((wn ? wn[e] : 1.0) * g[(int64_t)e * D + i], g[(int64_t)e * D + j], gn);
            }
            const double v = a + gn;
            hess[pt * D * D + i * D + j] = v;
            hess[pt * D * D + j * D + i] = v;
        }
        __syncthreads();
    }
}

// Launch of k_cost_hess over n points: as many points per CTA as fill its 256 threads with upper-triangle entries, within
// 48 KB of shared memory (at least one point: a forward cost of 96 emulators at D = 256 takes 194 KB).
int cost_hess(const double* mu, const double* obs, int64_t obs_ld, const double* weights, const double* s, const double* C,
              const double* deriv, const double* hs, int64_t n, int E, int D, int sms, double* hess, cudaStream_t st,
              bool pw = false, int64_t w_ld = 0) {
    const int nt = D * (D + 1) / 2;
    const size_t per = (size_t)E * (C ? 1 + D : 1);
    const int P = (int)std::max<size_t>(1, std::min<size_t>(std::max(1, 256 / nt), ((size_t)48 << 10) / (per * 8)));
    const size_t smem = (size_t)P * per * 8;
    if (smem > kSmemMax) return fail(GPE_ERR_UNSUPPORTED, "cost Hessian: %zu bytes of shared memory per point", smem);
    const int grid = (int)std::min<int64_t>((n + P - 1) / P, (int64_t)sms * 8);
    CUDA_TRY(launch_kernel(pw ? k_cost_hess<true> : k_cost_hess<false>, grid, 256, smem, st, mu, obs, obs_ld, weights, s, C, deriv,
                           hs, n, E, D, P, hess, w_ld));
    return GPE_OK;
}

// The chunk walk of the bank's cost calls on `st`: the bank means (and, with `grad`, their input gradients) of whole
// waves of 64-point tiles, at most 256 MB of them, go to the bank's cost scratch, and reduce(aux, mu, deriv, hs, ext, n0, n)
// consumes each chunk.  The scratch starts with aux_n doubles that the reducer may fill with per-call operands.  With
// `hess`, a second pass after the unchanged first one fills hs (n, E, D, D) (and deriv, if the first pass did not), and ext
// holds ext_pp doubles per point for the reducer: cost and gradient are those of the same call without `hess`.  A 64-point
// chunk is allocated even where it exceeds the 256 MB (wide Hessians: 96 emulators at D = 256).
template <typename Reduce>
int bank_cost_walk(gpe_bank* b, const double* testing, int64_t N, bool grad, bool hess, int64_t aux_n, int64_t ext_pp,
                   cudaStream_t st, int64_t call_N, Reduce reduce) {
    if (call_N < 0) call_N = N;
    const int64_t E = b->E, D = b->D;
    const int64_t per_point = E * (1 + (grad || hess ? D : 0)) + (hess ? E * D * D + ext_pp : 0);
    // points per chunk: whole waves of 64-point tiles, scratch bounded by 256 MB
    int64_t chunk = std::max<int64_t>(64, (((int64_t)256 << 20) / (per_point * 8)) / 64 * 64);
    chunk = std::min(chunk, (N + 63) / 64 * 64);
    const size_t need = (size_t)(aux_n + chunk * per_point);
    std::lock_guard<std::mutex> lock(b->cost_mu);
    if (!b->cost_free) CUDA_TRY(cudaEventCreateWithFlags(&b->cost_free, cudaEventDisableTiming));
    // the scratch may still be read by a reduction enqueued on another stream
    CUDA_TRY(cudaStreamWaitEvent(st, b->cost_free, 0));
    if (b->cost_cap < need) {
        if (b->cost_d) {
            CUDA_TRY(cudaEventSynchronize(b->cost_free));
            CUDA_TRY(cudaFree(b->cost_d));
            b->cost_d = nullptr; b->cost_cap = 0;
        }
        CUDA_TRY(cudaMalloc((void**)&b->cost_d, need * 8));
        b->cost_cap = need;
    }
    double* aux = b->cost_d;
    double* d_mu = b->cost_d + aux_n;
    double* d_der = grad || hess ? d_mu + chunk * E : nullptr;
    double* d_hes = hess ? d_der + chunk * E * D : nullptr;
    double* d_ext = hess ? d_hes + chunk * E * D * D : nullptr;
    for (int64_t n0 = 0; n0 < N; n0 += chunk) {
        const int64_t n = std::min(chunk, N - n0);
        int rc = bank_predict_device(b, testing + n0 * D, n, d_mu, nullptr, grad ? d_der : nullptr, nullptr, st, call_N);
        if (rc == GPE_OK && hess)
            rc = bank_predict_device(b, testing + n0 * D, n, nullptr, nullptr, grad ? nullptr : d_der, d_hes, st, call_N);
        if (rc == GPE_OK) rc = reduce(aux, d_mu, d_der, d_hes, d_ext, n0, n);
        if (rc) return rc;
    }
    CUDA_TRY(cudaEventRecord(b->cost_free, st));
    return GPE_OK;
}

// The cost calls take weights (K) shared by every point (w_ld = 0, or NULL: all 1) or one row per point, w_ld apart
// (DESIGN 4.6f).  Cn: NULL, or (spectrum cost with per-point weights and hess) the curvature C_n (N, E, E) of the points,
// formed beforehand by forward_cost_curv_pw (the solver keeps it across iterations).
int bank_cost_device(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld, const double* weights,
                     int64_t w_ld, const double*, double* cost, double* grad, double* hess, cudaStream_t st, int64_t call_N = -1) {
    const int64_t E = b->E, D = b->D;
    const int sms = b->models[0]->sms;
    const bool pw = w_ld != 0;
    return bank_cost_walk(b, testing, N, grad != nullptr, hess != nullptr, 0, 0, st, call_N,
                          [&](double*, const double* d_mu, const double* d_der, const double* d_hes, double*, int64_t n0,
                              int64_t n) -> int {
                              const double* w = pw ? weights + n0 * w_ld : weights;
                              if (cost || grad) {
                                  const int grid = (int)std::min<int64_t>((n + 3) / 4, (int64_t)sms * 16);
                                  CUDA_TRY(launch_kernel(pw ? k_bank_cost<true> : k_bank_cost<false>, grid, 128, (size_t)4 * E * 8,
                                                         st, d_mu, d_der, obs + n0 * obs_ld, obs_ld, w, cost ? cost + n0 : nullptr,
                                                         grad ? grad + n0 * D : nullptr, n, (int)E, (int)D, w_ld));
                              }
                              if (!hess) return GPE_OK;
                              return cost_hess(d_mu, obs + n0 * obs_ld, obs_ld, w, nullptr, nullptr, d_der, d_hes, n, (int)E,
                                               (int)D, sms, hess + n0 * D * D, st, pw, w_ld);
                          });
}

// Misfit of the back-projected spectra against observed ones (k_forward_cost, project.cu): the same walk, the spectra and
// Jacobians exist only as tiles inside the kernel.  The weights and the shared observation go to the scratch once per
// call, zero-padded to the basis image's width.
//   With hess, k_forward_cost also stores s = (l o (fwd - obs)) . basis^T (n, E) in the chunk scratch, and C = basis .
// diag(l) . basis^T (E, E) follows the partial sums in the aux area, formed once per call: the Gauss-Newton term G^T C G
// then costs E^2 D + E D^2 per point instead of D^2 W.  With per-point weights C_n is one (E, E) matrix per point: taken
// from Cn, or formed per chunk behind s in the chunk scratch.
int bank_forward_cost_device(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                             const double* weights, int64_t w_ld, const double* Cn, double* cost, double* grad, double* hess,
                             cudaStream_t st, int64_t call_N = -1) {
    const int D = b->D, W = b->W, Wp = b->Wp, E = b->E;
    const bool pw = w_ld != 0;
    // calls of a few points spread the column groups over CTAs; their partial sums follow the aux operands in the scratch
    const int gy = forward_cost_split(call_N < 0 ? N : call_N, W);
    const int64_t part_n = gy > 1 ? (int64_t)gy * ((N + 63) / 64 * 64) * (1 + E) : 0;
    const int64_t aux_n = 2 * (int64_t)Wp + part_n + (hess && !pw ? (int64_t)E * E : 0);
    const int64_t ext_pp = E + (hess && pw && !Cn ? (int64_t)E * E : 0);
    return bank_cost_walk(b, testing, N, grad != nullptr, hess != nullptr, aux_n, ext_pp, st, call_N,
                          [&](double* aux, const double* d_mu, const double* d_der, const double* d_hes, double* d_s,
                              int64_t n0, int64_t n) -> int {
                              const double* C = hess && !pw ? aux + 2 * Wp + part_n : nullptr;
                              const double* w = pw ? weights + n0 * w_ld : nullptr;
                              if (n0 == 0) CUDA_TRY(forward_cost_aux(pw ? nullptr : weights, obs_ld == 0 ? obs : nullptr, W, Wp, aux, st));
                              if (n0 == 0 && hess && !pw) CUDA_TRY(forward_cost_curv(b->d_basis, aux, E, Wp, (double*)C, st));
                              CUDA_TRY(forward_cost_rows(d_mu, d_der, n, E, D, obs + n0 * obs_ld, obs_ld, aux, b->d_basis, W,
                                                         Wp, gy, aux + 2 * Wp, cost ? cost + n0 : nullptr,
                                                         grad ? grad + n0 * D : nullptr, d_s, st, w, w_ld));
                              if (!hess) return GPE_OK;
                              if (pw && Cn) {
                                  C = Cn + n0 * E * E;
                              } else if (pw) {
                                  double* Cc = d_s + n * E;
                                  CUDA_TRY(forward_cost_curv_pw(b->d_basis, w, w_ld, n, E, W, Wp, Cc, st));
                                  C = Cc;
                              }
                              return cost_hess(nullptr, nullptr, 0, nullptr, d_s, C, d_der, d_hes, n, E, D, b->models[0]->sms,
                                               hess + n0 * D * D, st, pw, 0);
                          });
}

// Bank: testing in; mu, var, deriv, hess, fwd, deriv_full out (idx 0-5).  The PC means / gradients a projection consumes
// stay on the device as chunk intermediates (host NULL) when the caller did not ask for them.
CallIo bank_io(const gpe_bank* b, const double* testing, double* mu, double* var, double* deriv, double* hess, double* fwd,
               double* deriv_full) {
    const int64_t E = b->E, D = b->D, W = b->W;
    CallIo io;
    io.in.add(testing, D);
    io.idx[0] = (mu || fwd) ? io.out.add(mu, E) : -1;
    io.idx[1] = var ? io.out.add(var, E) : -1;
    io.idx[2] = (deriv || deriv_full) ? io.out.add(deriv, E * D) : -1;
    io.idx[3] = hess ? io.out.add(hess, E * D * D) : -1;
    io.idx[4] = fwd ? io.out.add(fwd, W) : -1;
    io.idx[5] = deriv_full ? io.out.add(deriv_full, D * W) : -1;
    return io;
}

// Host-resident bank call through the streaming pipeline: any of the point-major bank outputs plus the back-projected
// spectra / Jacobians.  Caller holds b->host_mu.
int bank_stream(gpe_bank* b, int64_t N, const CallIo& io, const SharedCall* shared = nullptr) {
    return stream_call(b->slots, b->device, b->models[0]->sms, io, N, 8, shared,
                       [&](int64_t, int64_t n, void* const* di, void* const* dout, cudaStream_t st) {
                           double *mu = io.at<double>(dout, 0), *deriv = io.at<double>(dout, 2);
                           double *fwd = io.at<double>(dout, 4), *deriv_full = io.at<double>(dout, 5);
                           int r = bank_predict_device(b, (const double*)di[0], n, mu, io.at<double>(dout, 1), deriv,
                                                       io.at<double>(dout, 3), st, N);
                           if (r == GPE_OK && (fwd || deriv_full)) r = bank_project_device(b, mu, deriv, n, fwd, deriv_full, st);
                           return r;
                       });
}

// Bank cost of observations K wide (E: the bank's own outputs, W: its spectra): testing and, unless obs_ld = 0, the
// per-point observations (idx 0) in; cost, grad, hess out (idx 1, 2, 3); per-point weights (w_ld != 0) in (idx 4).
CallIo cost_io(const gpe_bank* b, int64_t K, const double* testing, const double* obs, int64_t obs_ld, double* cost, double* grad,
               double* hess, const double* weights = nullptr, int64_t w_ld = 0) {
    CallIo io;
    io.in.add(testing, b->D);
    io.idx[0] = obs_ld != 0 ? io.in.add(obs, K) : -1;
    io.idx[4] = w_ld != 0 ? io.in.add(weights, K) : -1;
    io.idx[1] = cost ? io.out.add(cost, 1) : -1;
    io.idx[2] = grad ? io.out.add(grad, b->D) : -1;
    io.idx[3] = hess ? io.out.add(hess, (int64_t)b->D * b->D) : -1;
    return io;
}

typedef int (*CostDevice)(gpe_bank*, const double*, int64_t, const double*, int64_t, const double*, int64_t, const double*,
                          double*, double*, double*, cudaStream_t, int64_t);

// Host-resident cost call (bank_cost_device or bank_forward_cost_device, observations K wide): test points (and
// per-point observations) stream in, cost / gradient / Hessian stream out.
int bank_cost_stream(gpe_bank* b, int64_t K, CostDevice cost_device, int64_t N, const double* obs, int64_t obs_ld,
                     const double* weights, const CallIo& io, const SharedCall* shared = nullptr, int64_t w_ld = 0) {
    if (obs_ld != 0 && obs_ld != K) return fail(GPE_ERR_INVALID, "host observations must be contiguous: obs_ld = %s or 0", K == b->E ? "E" : "W");
    if (w_ld != 0 && w_ld != K) return fail(GPE_ERR_INVALID, "host weights must be contiguous: weights_ld = %s or 0", K == b->E ? "E" : "W");
    if (w_ld != 0) weights = nullptr;   // streamed per chunk (idx 4), not uploaded
    // the shared observation vector and the weights are small: one upload per call, enqueued ahead of this pipeline's first
    // chunk; its later chunks (other slot streams) wait for it.  (Every chunk of the previous call has finished: the
    // buffer is free.)
    const size_t aux_n = (size_t)(obs_ld == 0 ? K : 0) + (weights ? K : 0);
    double *d_obs1 = nullptr, *d_w = nullptr;
    if (aux_n > 0) {
        int rc = ensure_buf((void**)&b->d_aux, &b->aux_cap, aux_n * 8, false);
        if (rc) return rc;
        if (!b->aux_ready) CUDA_TRY(cudaEventCreateWithFlags(&b->aux_ready, cudaEventDisableTiming));
        d_obs1 = obs_ld == 0 ? b->d_aux : nullptr;
        d_w = weights ? b->d_aux + (obs_ld == 0 ? K : 0) : nullptr;
    }
    bool uploaded = false;
    return stream_call(b->slots, b->device, b->models[0]->sms, io, N, 8, shared,
                       [&](int64_t, int64_t n, void* const* di, void* const* dout, cudaStream_t st) {
                           if (aux_n > 0 && !uploaded) {
                               if (d_obs1) CUDA_TRY(cudaMemcpyAsync(d_obs1, obs, (size_t)K * 8, cudaMemcpyHostToDevice, st));
                               if (d_w) CUDA_TRY(cudaMemcpyAsync(d_w, weights, (size_t)K * 8, cudaMemcpyHostToDevice, st));
                               CUDA_TRY(cudaEventRecord(b->aux_ready, st));
                               uploaded = true;
                           } else if (aux_n > 0) {
                               CUDA_TRY(cudaStreamWaitEvent(st, b->aux_ready, 0));
                           }
                           const double* d_obs = obs_ld != 0 ? io.at<const double>(di, 0) : d_obs1;
                           const double* d_wc = w_ld != 0 ? io.at<const double>(di, 4) : d_w;
                           return cost_device(b, (const double*)di[0], n, d_obs, obs_ld != 0 ? K : 0, d_wc, w_ld != 0 ? K : 0,
                                              nullptr, io.at<double>(dout, 1), io.at<double>(dout, 2), io.at<double>(dout, 3), st, N);
                       });
}

// Request check of the weights of a call with observations K wide: w_ld = 0 (one shared row, or NULL), else per point,
// >= K apart on the device and exactly K for host arrays.
int weights_check(const double* weights, int64_t w_ld, int64_t K, bool spectra, bool host) {
    if (w_ld != 0 && !weights) return fail(GPE_ERR_INVALID, "weights_ld = %lld but weights is NULL", (long long)w_ld);
    if (w_ld != 0 && (w_ld < 0 || (host ? w_ld != K : w_ld < K)))
        return fail(GPE_ERR_INVALID, "weights_ld must be 0 (one weight vector) or %s %s", host ? "=" : ">=", spectra ? "W" : "E");
    return GPE_OK;
}

// Request check of the forward-cost calls (device: obs_ld = 0 or >= W; the host calls check obs_ld = 0 or W).
int forward_cost_check(gpe_bank* b, int64_t N, const double* testing, const double* obs, int64_t obs_ld, const double* cost,
                       const double* grad, const double* hess) {
    if (!b) return fail(GPE_ERR_INVALID, "bank is NULL");
    if (N < 0) return fail(GPE_ERR_INVALID, "N must be >= 0");
    if (!b->d_basis) return fail(GPE_ERR_INVALID, "bank was created without basis functions");
    if (!cost && !grad && !hess) return fail(GPE_ERR_INVALID, "no output requested");
    if (N > 0 && (!testing || !obs)) return fail(GPE_ERR_INVALID, "testing / obs is NULL");
    if (obs_ld != 0 && obs_ld < b->W) return fail(GPE_ERR_INVALID, "obs_ld must be 0 (one observed spectrum) or >= W");
    if (forward_cost_smem(b->E) > kSmemMax)
        return fail(GPE_ERR_UNSUPPORTED, "the forward cost supports banks of up to 96 emulators (got %d)", b->E);
    return GPE_OK;
}

// ---- candidate search (DESIGN 4.6e): kernels in search.cu ---------------------------------------------------------
// The search scratch of a call: the candidate table (built once per call) followed by the per-pixel work area of at most
// P pixels at a time.
constexpr int64_t kSearchRows = 1 << 16;
struct SearchScratch {
    int Kp = 0, gy = 1, Ew = 0;   // Ew: width of the ranking operand (E, or that of the per-point-weight forms)
    bool pw = false;
    int64_t P = 0;
    double *tbl = nullptr, *ta = nullptr, *mu = nullptr, *aux = nullptr, *C = nullptr;   // table (aux, C: spectrum cost)
    double *s = nullptr, *zeros = nullptr, *pv = nullptr, *x = nullptr, *cst = nullptr;   // pixels
    double *op = nullptr, *Cn = nullptr;                                                  // pixels, per-point weights
    int* pi = nullptr;
    int64_t* sel = nullptr;
};

// Width of the ranking operand of a search (DESIGN 4.6e, 4.6f).
int search_width(int E, bool spectra, bool pw) { return !pw ? E : spectra ? E * (E + 1) / 2 + E : 2 * E; }

// Lay out and grow the bank's search scratch for a call of call_N pixels (caller holds search_mu).
int search_prepare(gpe_bank* b, bool spectra, int64_t K, int k, int64_t call_N, SearchScratch* sc, bool pw = false) {
    const int64_t E = b->E, D = b->D;
    sc->Kp = search_pad(K);
    sc->gy = search_split(call_N, K);
    sc->P = std::min<int64_t>(kSearchRows, call_N);
    sc->pw = pw;
    sc->Ew = search_width((int)E, spectra, pw);
    const int64_t P = sc->P, gy = sc->gy, Ew = sc->Ew;
    size_t off = 0;
    auto carve = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_tbl = carve(8 * (size_t)search_ks((int)Ew) * sc->Kp * 4), o_ta = carve(8 * (size_t)sc->Kp), o_mu = carve(8 * K * E);
    const size_t o_aux = carve(spectra ? 16 * (size_t)b->Wp : 0), o_C = carve(spectra && !pw ? 8 * E * E : 0);
    const size_t o_s = carve(8 * P * E), o_z = carve(spectra ? 8 * P * E : 0), o_sel = carve(8 * P * k);
    const size_t o_pv = carve(gy > 1 ? 8 * gy * P * k : 0), o_pi = carve(gy > 1 ? 4 * gy * P * k : 0);
    const size_t o_x = carve(8 * P * D), o_cst = carve(8 * P * k);
    const size_t o_op = carve(pw ? 8 * P * Ew : 0), o_Cn = carve(pw && spectra ? 8 * P * E * E : 0);
    if (!b->search_free) CUDA_TRY(cudaEventCreateWithFlags(&b->search_free, cudaEventDisableTiming));
    if (b->search_cap < off) CUDA_TRY(cudaEventSynchronize(b->search_free));   // the old scratch may still be in use
    int rc = ensure_buf(&b->search_d, &b->search_cap, off, false);
    if (rc) return rc;
    char* base = (char*)b->search_d;
    sc->tbl = (double*)(base + o_tbl); sc->ta = (double*)(base + o_ta); sc->mu = (double*)(base + o_mu);
    sc->aux = spectra ? (double*)(base + o_aux) : nullptr; sc->C = spectra ? (double*)(base + o_C) : nullptr;
    sc->s = (double*)(base + o_s); sc->zeros = spectra ? (double*)(base + o_z) : nullptr; sc->sel = (int64_t*)(base + o_sel);
    sc->pv = (double*)(base + o_pv); sc->pi = (int*)(base + o_pi); sc->x = (double*)(base + o_x); sc->cst = (double*)(base + o_cst);
    sc->op = (double*)(base + o_op); sc->Cn = (double*)(base + o_Cn);
    return GPE_OK;
}

// Candidate table on st: the bank means at the K candidates (one call of K points), a_k and the packed image; for the
// spectrum cost also the padded weights / shared observation (aux) and C = basis . diag(l) . basis^T.
int search_build_table(gpe_bank* b, const SearchScratch& sc, bool spectra, const double* cand, int64_t K, const double* weights,
                       const double* obs1, cudaStream_t st) {
    const int E = b->E;
    int rc = bank_predict_device(b, cand, K, sc.mu, nullptr, nullptr, nullptr, st, K);
    if (rc) return rc;
    if (spectra) {
        CUDA_TRY(forward_cost_aux(sc.pw ? nullptr : weights, obs1, b->W, b->Wp, sc.aux, st));
        if (!sc.pw) CUDA_TRY(forward_cost_curv(b->d_basis, sc.aux, E, b->Wp, sc.C, st));
        CUDA_TRY(cudaMemsetAsync(sc.zeros, 0, (size_t)sc.P * E * 8, st));
    }
    if (sc.pw) CUDA_TRY(search_table_pw(sc.mu, K, E, sc.Ew, sc.Kp, spectra, sc.tbl, sc.ta, st));
    else CUDA_TRY(search_table(sc.mu, K, E, sc.Kp, spectra ? nullptr : weights, sc.C, sc.tbl, sc.ta, st));
    return GPE_OK;
}

// Pixels [0, n) of a call of call_N pixels on st, P at a time: pixel operand s (spectrum cost: s of k_forward_cost at
// fwd = 0, i.e. -basis . (l o obs)), top-k selection, then per slot j the exact cost of candidate sel[:, j] by the cost
// call's own path (call_N: the same kernel plans as a cost call of the call's pixels), then the final order.  Per-point
// weights (w_ld != 0): the operand of DESIGN 4.6f, from s and (spectrum cost) the pixels' curvature C_n.
int search_rows(gpe_bank* b, const SearchScratch& sc, bool spectra, const double* cand, int k, const double* obs, int64_t obs_ld,
                const double* weights, int64_t n, int64_t call_N, int64_t* idx, double* cost, cudaStream_t st, int64_t w_ld = 0) {
    const int E = b->E, D = b->D;
    const CostDevice cost_device = spectra ? bank_forward_cost_device : bank_cost_device;
    for (int64_t p0 = 0; p0 < n; p0 += sc.P) {
        const int64_t m = std::min(sc.P, n - p0);
        const double* o = obs + p0 * obs_ld;
        const double* w = w_ld != 0 ? weights + p0 * w_ld : weights;
        if (spectra)
            CUDA_TRY(forward_cost_rows(sc.zeros, nullptr, m, E, D, o, obs_ld, sc.aux, b->d_basis, b->W, b->Wp, 1, nullptr, nullptr,
                                       nullptr, sc.s, st, w_ld != 0 ? w : nullptr, w_ld));
        else if (w_ld == 0)
            CUDA_TRY(search_band_s(o, obs_ld, weights, m, E, sc.s, st));
        if (w_ld != 0 && spectra) CUDA_TRY(forward_cost_curv_pw(b->d_basis, w, w_ld, m, E, b->W, b->Wp, sc.Cn, st));
        if (w_ld != 0) CUDA_TRY(search_operand_pw(o, obs_ld, w, w_ld, sc.s, sc.Cn, m, E, sc.Ew, spectra, sc.op, st));
        CUDA_TRY(search_topk(w_ld != 0 ? sc.op : sc.s, m, sc.Ew, sc.tbl, sc.ta, sc.Kp, k, sc.gy, sc.pv, sc.pi, sc.sel, st));
        for (int j = 0; j < k; ++j) {
            CUDA_TRY(search_gather(cand, D, sc.sel, k, j, m, sc.x, st));
            int rc = cost_device(b, sc.x, m, o, obs_ld, w, w_ld, nullptr, sc.cst + (int64_t)j * m, nullptr, nullptr, st, call_N);
            if (rc) return rc;
        }
        CUDA_TRY(search_output(sc.sel, sc.cst, m, k, idx ? idx + p0 * k : nullptr, cost ? cost + p0 * k : nullptr, st));
    }
    return GPE_OK;
}

// Request check of the search calls (device: obs_ld = 0 or >= the observation width; host: 0 or equal to it).
int search_check(gpe_bank* b, const double* cand, int64_t K, const double* obs, int64_t N, int64_t obs_ld, int k,
                 const int64_t* idx, const double* cost, unsigned flags, bool host, const double* weights = nullptr,
                 int64_t w_ld = 0) {
    if (!b) return fail(GPE_ERR_INVALID, "bank is NULL");
    if (flags & ~(GPE_SOLVE_SPECTRA | GPE_HOST_PTRS)) return fail(GPE_ERR_INVALID, "unknown flag bits 0x%x", flags);
    const bool spectra = flags & GPE_SOLVE_SPECTRA;
    if (N < 0) return fail(GPE_ERR_INVALID, "N must be >= 0");
    if (K < 1 || K > ((int64_t)1 << 30)) return fail(GPE_ERR_INVALID, "K must be in [1, 2^30] (got %lld)", (long long)K);
    if (k < 1 || k > GPE_SEARCH_MAX_K || k > K)
        return fail(GPE_ERR_INVALID, "k must be in [1, min(K, %d)] (got %d)", GPE_SEARCH_MAX_K, k);
    if (spectra && !b->d_basis) return fail(GPE_ERR_INVALID, "bank was created without basis functions");
    const int64_t Kw = spectra ? b->W : b->E;
    if (obs_ld != 0 && (host ? obs_ld != Kw : obs_ld < Kw))
        return fail(GPE_ERR_INVALID, "obs_ld must be 0 (one observation) or %s %s", host ? "=" : ">=", spectra ? "W" : "E");
    if (!cand) return fail(GPE_ERR_INVALID, "cand is NULL");
    if (N > 0 && !obs) return fail(GPE_ERR_INVALID, "obs is NULL");
    if (!idx && !cost) return fail(GPE_ERR_INVALID, "no output requested");
    if (search_smem(b->E) > kSmemMax || (spectra && forward_cost_smem(b->E) > kSmemMax) || b->E > 96)
        return fail(GPE_ERR_UNSUPPORTED, "the search supports banks of up to 96 emulators (got %d)", b->E);
    int rc = weights_check(weights, w_ld, Kw, spectra, host);
    if (rc) return rc;
    if (w_ld != 0 && search_width(b->E, spectra, true) > 96)
        return fail(GPE_ERR_UNSUPPORTED, "with per-point weights the %s search supports banks of up to %d emulators (got %d)",
                    spectra ? "spectrum" : "band", spectra ? GPE_SEARCH_PW_MAX_E_SPECTRA : GPE_SEARCH_PW_MAX_E_BANDS, b->E);
    return GPE_OK;
}

// The streamed arrays of a host-resident search: per-point observations (unless shared) in; idx and cost (k 8-byte
// columns each) out.
CallIo search_io(int64_t Kw, const double* obs, int64_t obs_ld, int k, int64_t* idx, double* cost, const double* weights = nullptr,
                 int64_t w_ld = 0) {
    CallIo io;
    io.idx[0] = obs_ld != 0 ? io.in.add(obs, Kw) : -1;
    io.idx[3] = w_ld != 0 ? io.in.add(weights, Kw) : -1;
    io.idx[1] = idx ? io.out.add(idx, k) : -1;
    io.idx[2] = cost ? io.out.add(cost, k) : -1;
    return io;
}

// Host-resident search through the bank's pipeline (caller holds b->host_mu): the candidates and the shared operands are
// uploaded and the table is built once per call, then every chunk of pixels is searched on its slot's stream.  The
// chunks share the per-pixel scratch: each waits for the previous one through search_free.
int bank_search_stream(gpe_bank* b, bool spectra, const double* cand, int64_t K, const double* obs, int64_t N, int64_t obs_ld,
                       const double* weights, int k, const CallIo& io, const SharedCall* shared = nullptr, int64_t w_ld = 0) {
    const int64_t D = b->D, Kw = spectra ? b->W : b->E;
    struct Part { const double* src; int64_t n; double* dev; };
    Part parts[] = {{cand, K * D, nullptr}, {obs_ld == 0 ? obs : nullptr, Kw, nullptr}, {w_ld == 0 ? weights : nullptr, Kw, nullptr}};
    size_t total = 0;
    for (const Part& p : parts) if (p.src) total += ((size_t)p.n + 31) & ~(size_t)31;
    int rc = ensure_buf((void**)&b->d_aux, &b->aux_cap, total * 8, false);
    if (rc) return rc;
    double* at = b->d_aux;
    for (Part& p : parts) {
        if (!p.src) continue;
        CUDA_TRY(cudaMemcpyAsync(at, p.src, (size_t)p.n * 8, cudaMemcpyHostToDevice, cudaStreamLegacy));
        p.dev = at;
        at += ((size_t)p.n + 31) & ~(size_t)31;
    }
    std::lock_guard<std::mutex> lock(b->search_mu);
    SearchScratch sc;
    rc = search_prepare(b, spectra, K, k, N, &sc, w_ld != 0);
    if (rc) return rc;
    CUDA_TRY(cudaStreamWaitEvent(cudaStreamLegacy, b->search_free, 0));
    rc = search_build_table(b, sc, spectra, parts[0].dev, K, parts[2].dev, parts[1].dev, cudaStreamLegacy);
    if (rc) return rc;
    CUDA_TRY(cudaEventRecord(b->search_free, cudaStreamLegacy));
    // (a copy from pageable memory may return before its DMA has landed: the chunks' streams are not ordered after the
    // legacy stream, the event orders them)
    return stream_call(b->slots, b->device, b->models[0]->sms, io, N, 8, shared,
                       [&](int64_t, int64_t n, void* const* di, void* const* dout, cudaStream_t st) -> int {
                           CUDA_TRY(cudaStreamWaitEvent(st, b->search_free, 0));
                           const double* o = obs_ld != 0 ? io.at<const double>(di, 0) : parts[1].dev;
                           const double* w = w_ld != 0 ? io.at<const double>(di, 3) : parts[2].dev;
                           int r = search_rows(b, sc, spectra, parts[0].dev, k, o, obs_ld != 0 ? Kw : 0, w, n, N,
                                               io.at<int64_t>(dout, 1), io.at<double>(dout, 2), st, w_ld != 0 ? Kw : 0);
                           if (r) return r;
                           CUDA_TRY(cudaEventRecord(b->search_free, st));
                           return GPE_OK;
                       });
}

// ---- inversion (DESIGN 4.6d): bounded Levenberg-Marquardt, kernels in invert.cu ------------------------------------
// Solve of N points on `st` (device arrays), in sub-chunks whose solver scratch stays within 256 MB.  Each iteration
// evaluates the active trial points with the call's cost (cost, gradient and Hessian; call_N: the kernel plans follow the
// call, never the active count), runs k_lm_step, compacts the active list in ascending order and reads its length back
// through page-locked memory; the trial rows (and per-point observation and weight rows, when the list shrank) of the
// survivors are gathered for the next evaluation.  Synchronous: returns when the outputs are written.
//   Per-point weights with the spectrum cost: C_n depends on the weights only, so it is formed once per sub-chunk (Cs,
// E^2 doubles a point) and gathered with the weight rows, never recomputed per iteration (DESIGN 4.6f).
int bank_solve_device(gpe_bank* b, CostDevice cost_device, int64_t K, const LmProblem& pb, const double* x0, int64_t N,
                      const double* obs, int64_t obs_ld, const double* weights, double* x, double* cost, double* grad,
                      double* hess, double* cov, int32_t* info, cudaStream_t st, int64_t call_N, int64_t w_ld = 0) {
    const int64_t D = b->D, R = lm_state_doubles((int)D), E = b->E;
    const bool pw = w_ld > 0, curv = pw && cost_device == bank_forward_cost_device;
    // doubles per point, lists and flag included
    const int64_t per = R + D * D + 2 * D + 1 + (obs_ld > 0 ? K : 0) + (pw ? K : 0) + (curv ? 2 * E * E : 0) + 2;
    int64_t sub = std::max<int64_t>(1, std::min<int64_t>(N, (((int64_t)256 << 20) / 8) / per));
    if (const char* e = getenv("GPE_SOLVE_SUB_POINTS")) sub = std::max<int64_t>(1, std::min<int64_t>(sub, atoll(e)));   // dev aid: force sub-chunks in tests
    const size_t temp = lm_select_temp(sub);
    size_t off = 0;
    auto carve = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_state = carve(8 * sub * R), o_xe = carve(8 * sub * D), o_fe = carve(8 * sub), o_ge = carve(8 * sub * D);
    const size_t o_he = carve(8 * sub * D * D), o_obs = carve(obs_ld > 0 ? 8 * sub * K : 0), o_l0 = carve(4 * sub);
    const size_t o_l1 = carve(4 * sub), o_flag = carve(4 * sub), o_cnt = carve(4), o_tmp = carve(temp);
    const size_t o_w = carve(pw ? 8 * sub * K : 0), o_cs = carve(curv ? 8 * sub * E * E : 0), o_cc = carve(curv ? 8 * sub * E * E : 0);
    std::lock_guard<std::mutex> lock(b->solve_mu);
    int rc = ensure_buf(&b->solve_d, &b->solve_cap, off, false);
    if (rc) return rc;
    if (!b->solve_count) CUDA_TRY(cudaMallocHost((void**)&b->solve_count, sizeof(int)));
    if (!b->solve_ev) CUDA_TRY(cudaEventCreateWithFlags(&b->solve_ev, cudaEventDisableTiming));
    char* base = (char*)b->solve_d;
    double* state = (double*)(base + o_state);
    double *xe = (double*)(base + o_xe), *fe = (double*)(base + o_fe), *ge = (double*)(base + o_ge), *he = (double*)(base + o_he);
    double* obs_c = (double*)(base + o_obs);
    double *w_c = (double*)(base + o_w), *Cs = curv ? (double*)(base + o_cs) : nullptr, *C_c = (double*)(base + o_cc);
    int *lists[2] = {(int*)(base + o_l0), (int*)(base + o_l1)}, *flag = (int*)(base + o_flag), *d_cnt = (int*)(base + o_cnt);
    for (int64_t s0 = 0; s0 < N; s0 += sub) {
        const int64_t n = std::min(sub, N - s0);
        LmProblem p = pb;
        if (p.prior_mean && p.prior_ld > 0) p.prior_mean += s0 * p.prior_ld;
        const double* o = obs + s0 * obs_ld;
        const double* w = pw ? weights + s0 * w_ld : weights;
        CUDA_TRY(lm_init(p, x0 + s0 * D, n, state, xe, lists[0], st));
        if (curv) CUDA_TRY(forward_cost_curv_pw(b->d_basis, w, w_ld, n, (int)E, b->W, b->Wp, Cs, st));
        const double* e_obs = o;      // observation rows of the evaluation: the caller's while every point is active
        const double *e_w = w, *e_C = Cs;
        int64_t e_ld = obs_ld, e_wld = w_ld, act = n;
        for (int it = 0;; ++it) {
            int* list = lists[it & 1];
            int* next_list = lists[(it + 1) & 1];
            rc = cost_device(b, xe, act, e_obs, e_ld, e_w, e_wld, e_C, fe, ge, he, st, call_N);
            if (rc) return rc;
            CUDA_TRY(lm_step(p, act, list, fe, ge, he, state, flag, it == 0, st));
            CUDA_TRY(lm_select(list, flag, act, next_list, d_cnt, base + o_tmp, temp, st));
            CUDA_TRY(cudaMemcpyAsync(b->solve_count, d_cnt, sizeof(int), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaEventRecord(b->solve_ev, st));
            CUDA_TRY(cudaEventSynchronize(b->solve_ev));
            const int64_t next = *b->solve_count;
            if (next == 0) break;
            const bool regather = obs_ld > 0 && next < act;
            CUDA_TRY(lm_gather(state, (int)D, next_list, next, xe, o, regather ? obs_ld : 0, K, obs_c, st));
            if (regather) { e_obs = obs_c; e_ld = K; }
            if (pw && next < act) {
                CUDA_TRY(lm_gather_rows(next_list, next, w, w_ld, K, w_c, st));
                if (curv) CUDA_TRY(lm_gather_rows(next_list, next, Cs, E * E, E * E, C_c, st));
                e_w = w_c; e_wld = K; e_C = curv ? C_c : nullptr;
            }
            act = next;
        }
        CUDA_TRY(lm_output((int)D, n, state, x + s0 * D, cost ? cost + s0 : nullptr, grad ? grad + s0 * D : nullptr,
                           hess ? hess + s0 * D * D : nullptr, cov ? cov + s0 * D * D : nullptr, info + 2 * s0, st));
    }
    CUDA_TRY(cudaEventRecord(b->solve_ev, st));
    CUDA_TRY(cudaEventSynchronize(b->solve_ev));
    return GPE_OK;
}

// Solve of S series of T dates on `st` (device arrays; DESIGN 4.6g): bank_solve_device with series as the list entries.
// Each evaluation is act T rows of the call's cost (call_N: the call's row count), k_lm_series_step steps every active
// series, and the series that stay active are expanded into their rows for the row gathers of the point solver.  Scratch
// within 256 MB, in whole series.
int bank_series_solve_device(gpe_bank* b, CostDevice cost_device, int64_t K, const LmProblem& pb, const LmSeries& sp0,
                             const double* x0, int64_t S, const double* obs, int64_t obs_ld, const double* weights,
                             double* x, double* cost, double* grad, double* hess, double* cov, int32_t* info, cudaStream_t st,
                             int64_t call_N, int64_t w_ld = 0) {
    const int64_t D = b->D, R = lm_state_doubles((int)D), E = b->E, T = sp0.T;
    const bool pw = w_ld > 0, curv = pw && cost_device == bank_forward_cost_device;
    // doubles per series: per row those of the point solver (the row lists counted as a double), the block factors, and
    // the series list and flag
    const int64_t per_row = R + D * D + 2 * D + 1 + (obs_ld > 0 ? K : 0) + (pw ? K : 0) + (curv ? 2 * E * E : 0) + 2;
    const int64_t per = T * per_row + lm_series_scratch_doubles((int)D, (int)T) + 2;
    const int64_t cap = (((int64_t)256 << 20) / 8);
    if (per > cap)
        return fail(GPE_ERR_UNSUPPORTED, "one series of %lld dates needs %lld MB of solver scratch, beyond the 256 MB limit",
                    (long long)T, (long long)((per * 8) >> 20));
    int64_t sub = std::max<int64_t>(1, std::min<int64_t>(S, cap / per));
    if (const char* e = getenv("GPE_SOLVE_SUB_POINTS")) sub = std::max<int64_t>(1, std::min<int64_t>(sub, atoll(e)));   // dev aid: series here
    const int64_t rows_max = sub * T;
    const size_t temp = lm_select_temp(sub);
    size_t off = 0;
    auto carve = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_state = carve(8 * rows_max * R), o_xe = carve(8 * rows_max * D), o_fe = carve(8 * rows_max);
    const size_t o_ge = carve(8 * rows_max * D), o_he = carve(8 * rows_max * D * D), o_obs = carve(obs_ld > 0 ? 8 * rows_max * K : 0);
    const size_t o_l0 = carve(4 * rows_max), o_l1 = carve(4 * sub), o_rows = carve(4 * rows_max), o_flag = carve(4 * sub);
    const size_t o_cnt = carve(4), o_tmp = carve(temp), o_w = carve(pw ? 8 * rows_max * K : 0);
    const size_t o_cs = carve(curv ? 8 * rows_max * E * E : 0), o_cc = carve(curv ? 8 * rows_max * E * E : 0);
    const size_t o_scr = carve(8 * sub * lm_series_scratch_doubles((int)D, (int)T));
    std::lock_guard<std::mutex> lock(b->solve_mu);
    int rc = ensure_buf(&b->solve_d, &b->solve_cap, off, false);
    if (rc) return rc;
    if (!b->solve_count) CUDA_TRY(cudaMallocHost((void**)&b->solve_count, sizeof(int)));
    if (!b->solve_ev) CUDA_TRY(cudaEventCreateWithFlags(&b->solve_ev, cudaEventDisableTiming));
    char* base = (char*)b->solve_d;
    double* state = (double*)(base + o_state);
    double *xe = (double*)(base + o_xe), *fe = (double*)(base + o_fe), *ge = (double*)(base + o_ge), *he = (double*)(base + o_he);
    double* obs_c = (double*)(base + o_obs);
    double *w_c = (double*)(base + o_w), *Cs = curv ? (double*)(base + o_cs) : nullptr, *C_c = (double*)(base + o_cc);
    int *lists[2] = {(int*)(base + o_l0), (int*)(base + o_l1)}, *flag = (int*)(base + o_flag), *d_cnt = (int*)(base + o_cnt);
    int* rows = (int*)(base + o_rows);
    LmSeries sp = sp0;
    sp.scratch = (double*)(base + o_scr);
    for (int64_t s0 = 0; s0 < S; s0 += sub) {
        const int64_t n = std::min(sub, S - s0), r0 = s0 * T;
        LmProblem p = pb;
        if (p.prior_mean && p.prior_ld > 0) p.prior_mean += r0 * p.prior_ld;
        const double* o = obs + r0 * obs_ld;
        const double* w = pw ? weights + r0 * w_ld : weights;
        // lm_init numbers the rows: the first n entries of the list are then the series 0 .. n-1
        CUDA_TRY(lm_init(p, x0 + r0 * D, n * T, state, xe, lists[0], st));
        if (curv) CUDA_TRY(forward_cost_curv_pw(b->d_basis, w, w_ld, n * T, (int)E, b->W, b->Wp, Cs, st));
        const double* e_obs = o;
        const double *e_w = w, *e_C = Cs;
        int64_t e_ld = obs_ld, e_wld = w_ld, act = n;
        for (int it = 0;; ++it) {
            int* list = lists[it & 1];
            int* next_list = lists[(it + 1) & 1];
            rc = cost_device(b, xe, act * T, e_obs, e_ld, e_w, e_wld, e_C, fe, ge, he, st, call_N);
            if (rc) return rc;
            CUDA_TRY(lm_series_step(p, sp, act, list, fe, ge, he, state, flag, it == 0, st));
            CUDA_TRY(lm_select(list, flag, act, next_list, d_cnt, base + o_tmp, temp, st));
            CUDA_TRY(cudaMemcpyAsync(b->solve_count, d_cnt, sizeof(int), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaEventRecord(b->solve_ev, st));
            CUDA_TRY(cudaEventSynchronize(b->solve_ev));
            const int64_t next = *b->solve_count;
            if (next == 0) break;
            const bool regather = obs_ld > 0 && next < act;
            CUDA_TRY(lm_series_rows(next_list, next, (int)T, rows, st));
            CUDA_TRY(lm_gather(state, (int)D, rows, next * T, xe, o, regather ? obs_ld : 0, K, obs_c, st));
            if (regather) { e_obs = obs_c; e_ld = K; }
            if (pw && next < act) {
                CUDA_TRY(lm_gather_rows(rows, next * T, w, w_ld, K, w_c, st));
                if (curv) CUDA_TRY(lm_gather_rows(rows, next * T, Cs, E * E, E * E, C_c, st));
                e_w = w_c; e_wld = K; e_C = curv ? C_c : nullptr;
            }
            act = next;
        }
        CUDA_TRY(lm_series_output(p, sp, n, state, x + r0 * D, cost ? cost + s0 : nullptr, grad ? grad + r0 * D : nullptr,
                                  hess ? hess + r0 * D * D : nullptr, cov ? cov + r0 * D * D : nullptr, info + 2 * s0, st));
    }
    CUDA_TRY(cudaEventRecord(b->solve_ev, st));
    CUDA_TRY(cudaEventSynchronize(b->solve_ev));
    return GPE_OK;
}

constexpr gpe_solve_opts kSolveDefaults = {GPE_SOLVE_DEFAULT_MAX_ITER, 1e-10, 1e-10, 0.0, 1e-3, nullptr, nullptr, nullptr, 0, nullptr};

LmProblem lm_problem(int D, const gpe_solve_opts& o, const double* lower, const double* upper, const double* prior_mean,
                     int64_t prior_ld, const double* prior_prec) {
    return LmProblem{D, lower, upper, prior_mean, prior_ld, prior_prec, o.max_iter, o.ftol, o.xtol, o.gtol, o.lambda0};
}

// Request check of the solve calls; *o = the options with defaults for opts == NULL.  Reads the bounds (device pointers:
// a D2H copy on the call's stream `st`, so that it sees what the solve will read; the device is set).
int solve_check(gpe_bank* b, int64_t N, const double* x0, const double* obs, int64_t obs_ld, const gpe_solve_opts* opts,
                const double* x, const int32_t* info, unsigned flags, bool host, cudaStream_t st, gpe_solve_opts* o) {
    if (!b) return fail(GPE_ERR_INVALID, "bank is NULL");
    if (flags & ~(GPE_SOLVE_SPECTRA | GPE_HOST_PTRS)) return fail(GPE_ERR_INVALID, "unknown flag bits 0x%x", flags);
    if (N < 0) return fail(GPE_ERR_INVALID, "N must be >= 0");
    const bool spectra = flags & GPE_SOLVE_SPECTRA;
    const int D = b->D;
    const int64_t K = spectra ? b->W : b->E;
    if (spectra && !b->d_basis) return fail(GPE_ERR_INVALID, "bank was created without basis functions");
    *o = opts ? *opts : kSolveDefaults;
    if (o->max_iter < 0) return fail(GPE_ERR_INVALID, "max_iter must be >= 0");
    if (!(o->ftol >= 0 && o->xtol >= 0 && o->gtol >= 0 && o->lambda0 > 0))
        return fail(GPE_ERR_INVALID, "ftol, xtol, gtol must be >= 0 and lambda0 > 0");
    if (o->prior_mean && !o->prior_prec) return fail(GPE_ERR_INVALID, "prior_mean given without prior_prec");
    if (o->prior_mean && o->prior_ld != 0 && (host ? o->prior_ld != D : o->prior_ld < D))
        return fail(GPE_ERR_INVALID, "prior_ld must be 0 (one prior mean) or %s D", host ? "=" : ">=");
    if (obs_ld != 0 && (host ? obs_ld != K : obs_ld < K))
        return fail(GPE_ERR_INVALID, "obs_ld must be 0 (one observation) or %s %s", host ? "=" : ">=", spectra ? "W" : "E");
    if (N > 0 && (!x0 || !obs || !x || !info)) return fail(GPE_ERR_INVALID, "x0 / obs / x / info is NULL");
    if (D > GPE_SOLVE_MAX_D) return fail(GPE_ERR_UNSUPPORTED, "the solver supports D <= %d (got %d)", GPE_SOLVE_MAX_D, D);
    if (spectra && forward_cost_smem(b->E) > kSmemMax)
        return fail(GPE_ERR_UNSUPPORTED, "the forward cost supports banks of up to 96 emulators (got %d)", b->E);
    if (o->lower && o->upper) {
        double lo[GPE_SOLVE_MAX_D], hi[GPE_SOLVE_MAX_D];
        if (host) {
            memcpy(lo, o->lower, D * 8);
            memcpy(hi, o->upper, D * 8);
        } else {
            CUDA_TRY(cudaSetDevice(b->device));
            CUDA_TRY(cudaMemcpyAsync(lo, o->lower, D * 8, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaMemcpyAsync(hi, o->upper, D * 8, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
        }
        for (int d = 0; d < D; ++d)
            if (!(lo[d] <= hi[d])) return fail(GPE_ERR_INVALID, "lower[%d] > upper[%d] (or NaN)", d, d);
    }
    return GPE_OK;
}

// Request check of the series arguments (DESIGN 4.6g): S >= 0, T >= 1, R (D, D) finite and exactly symmetric, coupling
// (T - 1) finite and >= 0 or NULL.  Device pointers are read with a D2H copy on the call's stream `st`.
int series_check(gpe_bank* b, int64_t S, int64_t T, const double* R, const double* coupling, bool host, cudaStream_t st) {
    if (S < 0) return fail(GPE_ERR_INVALID, "S must be >= 0");
    if (T < 1 || T > (1 << 24)) return fail(GPE_ERR_INVALID, "T must be in [1, 2^24] (got %lld)", (long long)T);
    if (!R) return fail(GPE_ERR_INVALID, "smooth_prec is NULL");
    const int D = b->D;
    if (D > GPE_SOLVE_MAX_D) return fail(GPE_ERR_UNSUPPORTED, "the solver supports D <= %d (got %d)", GPE_SOLVE_MAX_D, D);
    std::vector<double> r((size_t)D * D), c(coupling ? (size_t)(T - 1) : 0);
    if (host) {
        memcpy(r.data(), R, r.size() * 8);
        if (!c.empty()) memcpy(c.data(), coupling, c.size() * 8);
    } else {
        CUDA_TRY(cudaSetDevice(b->device));
        CUDA_TRY(cudaMemcpyAsync(r.data(), R, r.size() * 8, cudaMemcpyDeviceToHost, st));
        if (!c.empty()) CUDA_TRY(cudaMemcpyAsync(c.data(), coupling, c.size() * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    for (int i = 0; i < D; ++i)
        for (int j = 0; j < D; ++j) {
            if (!std::isfinite(r[i * D + j])) return fail(GPE_ERR_INVALID, "smooth_prec[%d, %d] is not finite", i, j);
            if (r[i * D + j] != r[j * D + i]) return fail(GPE_ERR_INVALID, "smooth_prec is not symmetric at (%d, %d)", i, j);
        }
    for (size_t t = 0; t < c.size(); ++t)
        if (!(std::isfinite(c[t]) && c[t] >= 0.0)) return fail(GPE_ERR_INVALID, "coupling[%zu] must be finite and >= 0", t);
    return GPE_OK;
}

// The streamed arrays of a host-resident solve: x0 and, when per point, obs and the prior means in; x, the optional
// cost / grad / hess / cov and info (8 bytes a point: one double-wide column) out.
struct SolveIo {
    CallIo io;
    int obs = -1, w = -1, pm = -1, x = -1, cost = -1, grad = -1, hess = -1, cov = -1, info = -1;
};

// T > 1: the unit is a series of T rows (cost and info stay one per series).
SolveIo solve_io(int64_t D, int64_t K, const double* x0, const double* obs, int64_t obs_ld, const gpe_solve_opts& o, double* x,
                 double* cost, double* grad, double* hess, double* cov, int32_t* info, const double* weights = nullptr,
                 int64_t w_ld = 0, int64_t T = 1) {
    SolveIo s;
    s.io.in.add(x0, T * D);
    if (obs_ld != 0) s.obs = s.io.in.add(obs, T * K);
    if (w_ld != 0) s.w = s.io.in.add(weights, T * K);
    if (o.prior_mean && o.prior_ld != 0) s.pm = s.io.in.add(o.prior_mean, T * D);
    s.x = s.io.out.add(x, T * D);
    if (cost) s.cost = s.io.out.add(cost, 1);
    if (grad) s.grad = s.io.out.add(grad, T * D);
    if (hess) s.hess = s.io.out.add(hess, T * D * D);
    if (cov) s.cov = s.io.out.add(cov, T * D * D);
    s.info = s.io.out.add(info, 1);
    return s;
}

// Host-resident solve through the bank's pipeline (caller holds b->host_mu): the small per-call operands (shared
// observation, weights, bounds, shared prior mean, precision) are uploaded once, then every chunk is solved by
// bank_solve_device as its chunk launch.  A chunk's solve blocks this pipeline's thread until it has finished.
//   series (host R and coupling): N series, each chunk solved by bank_series_solve_device; R and coupling are uploaded too.
int bank_solve_stream(gpe_bank* b, bool spectra, int64_t N, const double* obs, int64_t obs_ld, const double* weights,
                      const gpe_solve_opts& o, const SolveIo& s, const SharedCall* shared = nullptr,
                      const LmSeries* series = nullptr) {
    const int64_t D = b->D, K = spectra ? b->W : b->E, T = series ? series->T : 1;
    struct Part { const double* src; int64_t n; double* dev; };
    Part parts[] = {{obs_ld == 0 ? obs : nullptr, K, nullptr}, {s.w < 0 ? weights : nullptr, K, nullptr}, {o.lower, D, nullptr},
                    {o.upper, D, nullptr}, {o.prior_ld == 0 ? o.prior_mean : nullptr, D, nullptr}, {o.prior_prec, D * D, nullptr},
                    {series ? series->R : nullptr, D * D, nullptr}, {series ? series->coupling : nullptr, T - 1, nullptr}};
    size_t total = 0;
    for (const Part& p : parts) if (p.src && p.n > 0) total += (size_t)p.n;
    if (total > 0) {
        int rc = ensure_buf((void**)&b->d_aux, &b->aux_cap, total * 8, false);
        if (rc) return rc;
        double* at = b->d_aux;
        for (Part& p : parts) {
            if (!p.src || p.n == 0) continue;
            CUDA_TRY(cudaMemcpyAsync(at, p.src, (size_t)p.n * 8, cudaMemcpyHostToDevice, cudaStreamLegacy));
            p.dev = at;
            at += p.n;
        }
        // The chunks run on the slots' non-blocking streams, which are not ordered after the legacy stream, and a copy from
        // pageable memory may return before its DMA has landed: wait for the copies here.
        CUDA_TRY(cudaStreamSynchronize(cudaStreamLegacy));
    }
    const LmProblem pb = lm_problem((int)D, o, parts[2].dev, parts[3].dev, parts[4].dev, 0, parts[5].dev);
    return stream_call(b->slots, b->device, b->models[0]->sms, s.io, N, 8, shared,
                       [&](int64_t, int64_t n, void* const* di, void* const* dout, cudaStream_t st) {
                           LmProblem p = pb;
                           if (s.pm >= 0) { p.prior_mean = (const double*)di[s.pm]; p.prior_ld = D; }
                           auto out = [&](int k) { return k >= 0 ? (double*)dout[k] : nullptr; };
                           if (series)
                               return bank_series_solve_device(
                                   b, spectra ? bank_forward_cost_device : bank_cost_device, K, p,
                                   LmSeries{(int)T, parts[7].dev, parts[6].dev, nullptr}, (const double*)di[0], n,
                                   s.obs >= 0 ? (const double*)di[s.obs] : parts[0].dev, obs_ld != 0 ? K : 0,
                                   s.w >= 0 ? (const double*)di[s.w] : parts[1].dev, out(s.x), out(s.cost), out(s.grad),
                                   out(s.hess), out(s.cov), (int32_t*)dout[s.info], st, N * T, s.w >= 0 ? K : 0);
                           return bank_solve_device(b, spectra ? bank_forward_cost_device : bank_cost_device, K, p,
                                                    (const double*)di[0], n, s.obs >= 0 ? (const double*)di[s.obs] : parts[0].dev,
                                                    obs_ld != 0 ? K : 0, s.w >= 0 ? (const double*)di[s.w] : parts[1].dev,
                                                    out(s.x), out(s.cost), out(s.grad), out(s.hess), out(s.cov),
                                                    (int32_t*)dout[s.info], st, N, s.w >= 0 ? K : 0);
                       });
}

int bank_check_outputs(gpe_bank* b, int64_t N, const double* testing, double*& mu, double*& var, double*& deriv, double*& hess,
                       double*& fwd, double*& deriv_full, unsigned flags) {
    if (!b) return fail(GPE_ERR_INVALID, "bank is NULL");
    if (N < 0) return fail(GPE_ERR_INVALID, "N must be >= 0");
    if (N > 0 && !testing) return fail(GPE_ERR_INVALID, "testing is NULL");
    int rc = take_outputs(flags, mu, var, deriv, hess, fwd, deriv_full);
    if (rc) return rc;
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

// One host-resident call on the devices of mm; run(owner, shared) streams an owner's share of it (caller holds the
// owner's host_mu; shared NULL: the whole call).  With one device, or up to solo_max points, the call is one chunk: the
// first device serves it on the calling thread (no thread fan-out, and the mapped-buffer path for the reference's
// one-point calls stays available) -- same kernels, same result; solo_max < 0 always fans out.  Otherwise one thread per
// device pulls the chunks of one shared plan from one cursor.  The kernel plan (tile size) follows the size of the whole
// call, so G devices reproduce one device bit for bit.
template <typename Owner, typename Run>
int fan_out(gpe_multi* mm, const std::vector<Owner*>& owners, int sms, const CallIo& io, int64_t N, int64_t solo_max, Run run) {
    const int G = (int)owners.size();
    if (solo_max >= 0 && (G == 1 || N <= solo_max)) {
        DeviceRestore restore_device;
        CUDA_TRY(cudaSetDevice(owners[0]->device));
        std::lock_guard<std::mutex> lock(owners[0]->host_mu);
        return run(owners[0], nullptr);
    }
    const StreamPlan pl = stream_plan(io, N, 8, sms, G);
    std::atomic<int64_t> cursor{0};
    ChunkSource src{&cursor, N, pl.CH};
    // large page-locked calls: decide (once per handle) whether some devices should send their host traffic through a
    // partner's PCIe link
    const bool relay_ok = pl.in_direct && pl.out_direct && N >= 4 * pl.CH;
    if (relay_ok) multi_route(mm);
    return run_per_device(G, mm->devices.data(), [&](int g) {
        Owner* o = owners[g];
        std::lock_guard<std::mutex> lock(o->host_mu);   // also guards the buffers of the device's relay
        int rc = GPE_OK;
        const Relay* relay = (relay_ok && mm->routed && !mm->relays.empty()) ? multi_relay(mm, g, pl, io.in, io.out, &rc) : nullptr;
        if (rc) return rc;
        const SharedCall shared{&pl, &src, relay};
        return run(o, &shared);
    });
}

// The cost calls of one bank (band cost, or spectra with GPE_SOLVE_SPECTRA; host arrays with GPE_HOST_PTRS).
int bank_cost_call(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld, const double* weights,
                   int64_t w_ld, double* cost, double* grad, double* hess, unsigned flags, void* stream) {
    const bool host = flags & GPE_HOST_PTRS, spectra = flags & GPE_SOLVE_SPECTRA;
    if (spectra) {
        int rc = forward_cost_check(b, N, testing, obs, obs_ld, cost, grad, hess);
        if (rc || N == 0) return rc;
    } else {
        if (!b) return fail(GPE_ERR_INVALID, "bank is NULL");
        if (N < 0) return fail(GPE_ERR_INVALID, "N must be >= 0");
        if (N == 0) return GPE_OK;
        if (!testing || !obs) return fail(GPE_ERR_INVALID, "testing / obs is NULL");
        if (!cost && !grad && !hess) return fail(GPE_ERR_INVALID, "no output requested");
        if (!host && obs_ld != 0 && obs_ld < b->E) return fail(GPE_ERR_INVALID, "obs_ld must be 0 (one observation vector) or >= E");
    }
    const int64_t K = spectra ? b->W : b->E;
    int rc = weights_check(weights, w_ld, K, spectra, host);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(b->device));
    const CostDevice cost_device = spectra ? bank_forward_cost_device : bank_cost_device;
    if (host) {
        std::lock_guard<std::mutex> lock(b->host_mu);
        return bank_cost_stream(b, K, cost_device, N, obs, obs_ld, weights,
                                cost_io(b, K, testing, obs, obs_ld, cost, grad, hess, weights, w_ld), nullptr, w_ld);
    }
    return cost_device(b, testing, N, obs, obs_ld, weights, w_ld, nullptr, cost, grad, hess, (cudaStream_t)stream, -1);
}

// The same on every device of a bank handle (host arrays).
int multi_bank_cost_call(gpe_multi* mm, const double* testing, int64_t N, const double* obs, int64_t obs_ld, const double* weights,
                         int64_t w_ld, double* cost, double* grad, double* hess, bool spectra) {
    if (!mm || mm->banks.empty()) return fail(GPE_ERR_INVALID, "handle is NULL or not a bank handle");
    gpe_bank* b0 = mm->banks[0];
    if (spectra) {
        int rc = forward_cost_check(b0, N, testing, obs, obs_ld, cost, grad, hess);
        if (rc || N == 0) return rc;
    } else {
        if (N < 0) return fail(GPE_ERR_INVALID, "N must be >= 0");
        if (N == 0) return GPE_OK;
        if (!testing || !obs) return fail(GPE_ERR_INVALID, "testing / obs is NULL");
        if (!cost && !grad && !hess) return fail(GPE_ERR_INVALID, "no output requested");
    }
    const int64_t K = spectra ? b0->W : b0->E;
    int rc = weights_check(weights, w_ld, K, spectra, true);
    if (rc) return rc;
    const CostDevice cost_device = spectra ? bank_forward_cost_device : bank_cost_device;
    const CallIo io = cost_io(b0, K, testing, obs, obs_ld, cost, grad, hess, weights, w_ld);
    return fan_out(mm, mm->banks, b0->models[0]->sms, io, N, -1, [&](gpe_bank* b, const SharedCall* shared) {
        return bank_cost_stream(b, K, cost_device, N, obs, obs_ld, weights, io, shared, w_ld);
    });
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
        const cudaError_t e = upload(&b->d_entries, ent);
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
                e = upload(&b->d_gx, gx);
            }
            if (e == cudaSuccess) e = upload(&b->d_galpha[grad], galpha);
            if (e == cudaSuccess) e = upload(&b->d_gw[grad], gw);
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
        const cudaError_t e = upload(&b->d_basis, bt);
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
    if (b->aux_ready) cudaEventDestroy(b->aux_ready);
    if (b->cost_d) cudaFree(b->cost_d);
    if (b->cost_free) cudaEventDestroy(b->cost_free);
    if (b->solve_d) cudaFree(b->solve_d);
    if (b->solve_count) cudaFreeHost(b->solve_count);
    if (b->solve_ev) cudaEventDestroy(b->solve_ev);
    if (b->search_d) cudaFree(b->search_d);
    if (b->search_free) cudaEventDestroy(b->search_free);
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
        return bank_stream(b, N, bank_io(b, testing, mu, var, deriv, hess, fwd, deriv_full));
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

int gpe_bank_cost_ex(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld, const double* weights,
                     double* cost, double* grad, double* hess, void* stream) {
    NvtxRange nvtx_range("gpe_bank_cost");
    return bank_cost_call(b, testing, N, obs, obs_ld, weights, 0, cost, grad, hess, 0u, stream);
}

int gpe_bank_cost_pw(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld, const double* weights,
                     int64_t weights_ld, double* cost, double* grad, double* hess, unsigned flags, void* stream) {
    NvtxRange nvtx_range("gpe_bank_cost_pw");
    if (flags & ~(GPE_SOLVE_SPECTRA | GPE_HOST_PTRS)) return fail(GPE_ERR_INVALID, "unknown flag bits 0x%x", flags);
    return bank_cost_call(b, testing, N, obs, obs_ld, weights, weights_ld, cost, grad, hess, flags, stream);
}

int gpe_bank_cost(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld, const double* weights,
                  double* cost, double* grad, void* stream) {
    return gpe_bank_cost_ex(b, testing, N, obs, obs_ld, weights, cost, grad, nullptr, stream);
}

int gpe_bank_cost_host_ex(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                          const double* weights, double* cost, double* grad, double* hess) {
    NvtxRange nvtx_range("gpe_bank_cost_host");
    return bank_cost_call(b, testing, N, obs, obs_ld, weights, 0, cost, grad, hess, GPE_HOST_PTRS, nullptr);
}

int gpe_bank_cost_host(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                       const double* weights, double* cost, double* grad) {
    return gpe_bank_cost_host_ex(b, testing, N, obs, obs_ld, weights, cost, grad, nullptr);
}

int gpe_bank_forward_cost_ex(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                             const double* weights, double* cost, double* grad, double* hess, void* stream) {
    NvtxRange nvtx_range("gpe_bank_forward_cost");
    return bank_cost_call(b, testing, N, obs, obs_ld, weights, 0, cost, grad, hess, GPE_SOLVE_SPECTRA, stream);
}

int gpe_bank_forward_cost(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                          const double* weights, double* cost, double* grad, void* stream) {
    return gpe_bank_forward_cost_ex(b, testing, N, obs, obs_ld, weights, cost, grad, nullptr, stream);
}

int gpe_bank_forward_cost_host_ex(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                                  const double* weights, double* cost, double* grad, double* hess) {
    NvtxRange nvtx_range("gpe_bank_forward_cost_host");
    return bank_cost_call(b, testing, N, obs, obs_ld, weights, 0, cost, grad, hess, GPE_SOLVE_SPECTRA | GPE_HOST_PTRS, nullptr);
}

int gpe_bank_forward_cost_host(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                               const double* weights, double* cost, double* grad) {
    return gpe_bank_forward_cost_host_ex(b, testing, N, obs, obs_ld, weights, cost, grad, nullptr);
}

int gpe_bank_solve_pw(gpe_bank* b, const double* x0, int64_t N, const double* obs, int64_t obs_ld, const double* weights,
                      int64_t weights_ld, const gpe_solve_opts* opts, double* x, double* cost, double* grad, double* hess,
                      double* cov, int32_t* info, unsigned flags, void* stream) {
    NvtxRange nvtx_range("gpe_bank_solve");
    const bool host = flags & GPE_HOST_PTRS, spectra = flags & GPE_SOLVE_SPECTRA;
    gpe_solve_opts o;
    int rc = solve_check(b, N, x0, obs, obs_ld, opts, x, info, flags, host, (cudaStream_t)stream, &o);
    if (rc == GPE_OK) rc = weights_check(weights, weights_ld, spectra ? b->W : b->E, spectra, host);
    if (rc || N == 0) return rc;
    CUDA_TRY(cudaSetDevice(b->device));
    const int64_t D = b->D, K = spectra ? b->W : b->E;
    if (host) {
        std::lock_guard<std::mutex> lock(b->host_mu);
        return bank_solve_stream(b, spectra, N, obs, obs_ld, weights, o,
                                 solve_io(D, K, x0, obs, obs_ld, o, x, cost, grad, hess, cov, info, weights, weights_ld));
    }
    const LmProblem pb = lm_problem((int)D, o, o.lower, o.upper, o.prior_mean, o.prior_ld, o.prior_prec);
    return bank_solve_device(b, spectra ? bank_forward_cost_device : bank_cost_device, K, pb, x0, N, obs, obs_ld, weights, x,
                             cost, grad, hess, cov, info, (cudaStream_t)stream, N, weights_ld);
}

int gpe_bank_solve(gpe_bank* b, const double* x0, int64_t N, const double* obs, int64_t obs_ld, const double* weights,
                   const gpe_solve_opts* opts, double* x, double* cost, double* grad, double* hess, double* cov,
                   int32_t* info, unsigned flags, void* stream) {
    return gpe_bank_solve_pw(b, x0, N, obs, obs_ld, weights, 0, opts, x, cost, grad, hess, cov, info, flags, stream);
}

int gpe_bank_solve_series(gpe_bank* b, int64_t S, int64_t T, const double* x0, const double* obs, int64_t obs_ld,
                          const double* weights, int64_t weights_ld, const gpe_solve_opts* opts, const double* smooth_prec,
                          const double* coupling, double* x, double* cost, double* grad, double* hess, double* cov,
                          int32_t* info, unsigned flags, void* stream) {
    NvtxRange nvtx_range("gpe_bank_solve_series");
    const bool host = flags & GPE_HOST_PTRS, spectra = flags & GPE_SOLVE_SPECTRA;
    if (!b) return fail(GPE_ERR_INVALID, "bank is NULL");
    int rc = series_check(b, S, T, smooth_prec, coupling, host, (cudaStream_t)stream);
    gpe_solve_opts o;
    if (rc == GPE_OK) rc = solve_check(b, S * T, x0, obs, obs_ld, opts, x, info, flags, host, (cudaStream_t)stream, &o);
    if (rc == GPE_OK) rc = weights_check(weights, weights_ld, spectra ? b->W : b->E, spectra, host);
    if (rc || S == 0) return rc;
    CUDA_TRY(cudaSetDevice(b->device));
    const int64_t D = b->D, K = spectra ? b->W : b->E;
    const LmSeries sp{(int)T, coupling, smooth_prec, nullptr};
    if (host) {
        std::lock_guard<std::mutex> lock(b->host_mu);
        return bank_solve_stream(b, spectra, S, obs, obs_ld, weights, o,
                                 solve_io(D, K, x0, obs, obs_ld, o, x, cost, grad, hess, cov, info, weights, weights_ld, T),
                                 nullptr, &sp);
    }
    const LmProblem pb = lm_problem((int)D, o, o.lower, o.upper, o.prior_mean, o.prior_ld, o.prior_prec);
    return bank_series_solve_device(b, spectra ? bank_forward_cost_device : bank_cost_device, K, pb, sp, x0, S, obs, obs_ld,
                                    weights, x, cost, grad, hess, cov, info, (cudaStream_t)stream, S * T, weights_ld);
}

int gpe_bank_search_pw(gpe_bank* b, const double* cand, int64_t K, const double* obs, int64_t N, int64_t obs_ld,
                       const double* weights, int64_t weights_ld, int k, int64_t* idx, double* cost, unsigned flags, void* stream) {
    NvtxRange nvtx_range("gpe_bank_search");
    const bool host = flags & GPE_HOST_PTRS, spectra = flags & GPE_SOLVE_SPECTRA;
    int rc = search_check(b, cand, K, obs, N, obs_ld, k, idx, cost, flags, host, weights, weights_ld);
    if (rc || N == 0) return rc;
    CUDA_TRY(cudaSetDevice(b->device));
    if (host) {
        std::lock_guard<std::mutex> lock(b->host_mu);
        return bank_search_stream(b, spectra, cand, K, obs, N, obs_ld, weights, k,
                                  search_io(spectra ? b->W : b->E, obs, obs_ld, k, idx, cost, weights, weights_ld), nullptr,
                                  weights_ld);
    }
    const cudaStream_t st = (cudaStream_t)stream;
    std::lock_guard<std::mutex> lock(b->search_mu);
    SearchScratch sc;
    rc = search_prepare(b, spectra, K, k, N, &sc, weights_ld != 0);
    if (rc) return rc;
    CUDA_TRY(cudaStreamWaitEvent(st, b->search_free, 0));
    rc = search_build_table(b, sc, spectra, cand, K, weights, obs_ld == 0 ? obs : nullptr, st);
    if (rc == GPE_OK) rc = search_rows(b, sc, spectra, cand, k, obs, obs_ld, weights, N, N, idx, cost, st, weights_ld);
    if (rc) return rc;
    CUDA_TRY(cudaEventRecord(b->search_free, st));
    return GPE_OK;
}

int gpe_bank_search(gpe_bank* b, const double* cand, int64_t K, const double* obs, int64_t N, int64_t obs_ld,
                    const double* weights, int k, int64_t* idx, double* cost, unsigned flags, void* stream) {
    return gpe_bank_search_pw(b, cand, K, obs, N, obs_ld, weights, 0, k, idx, cost, flags, stream);
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
    if (!testing) return fail(GPE_ERR_INVALID, "testing is NULL");
    int rc = take_outputs(flags, mu, var, deriv, hess);
    if (rc) return rc;
    gpe_model* m0 = mm->models[0];
    const CallIo io = model_io(m0->D, testing, mu, var, deriv, hess);
    return fan_out(mm, mm->models, m0->sms, io, N, 3 * 64 * (int64_t)m0->sms,
                   [&](gpe_model* m, const SharedCall* shared) { return model_stream(m, N, io, shared); });
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
        if (!testing[g]) return fail(GPE_ERR_INVALID, "testing[%d] is NULL", g);
        double *o_mu = mu ? mu[g] : nullptr, *o_var = var ? var[g] : nullptr;
        double *o_der = deriv ? deriv[g] : nullptr, *o_hes = hess ? hess[g] : nullptr;
        int rc = take_outputs(flags, o_mu, o_var, o_der, o_hes);
        if (rc) return rc;
        CUDA_TRY(cudaSetDevice(m->device));
        rc = predict_device(m, testing[g], N[g], o_mu, o_var, o_der, o_hes, 1, 1, m->D, (int64_t)m->D * m->D,
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
    const int sms = b0->models[0]->sms;
    const CallIo io = bank_io(b0, testing, mu, var, deriv, hess, fwd, deriv_full);
    return fan_out(mm, mm->banks, sms, io, N, 64 * (int64_t)sms,
                   [&](gpe_bank* b, const SharedCall* shared) { return bank_stream(b, N, io, shared); });
}

int gpe_multi_bank_cost_ex(gpe_multi* mm, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                           const double* weights, double* cost, double* grad, double* hess) {
    NvtxRange nvtx_range("gpe_multi_bank_cost");
    return multi_bank_cost_call(mm, testing, N, obs, obs_ld, weights, 0, cost, grad, hess, false);
}

int gpe_multi_bank_cost_pw(gpe_multi* mm, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                           const double* weights, int64_t weights_ld, double* cost, double* grad, double* hess, unsigned flags) {
    NvtxRange nvtx_range("gpe_multi_bank_cost_pw");
    if (flags & ~(GPE_SOLVE_SPECTRA | GPE_HOST_PTRS)) return fail(GPE_ERR_INVALID, "unknown flag bits 0x%x", flags);
    return multi_bank_cost_call(mm, testing, N, obs, obs_ld, weights, weights_ld, cost, grad, hess, flags & GPE_SOLVE_SPECTRA);
}

int gpe_multi_bank_cost(gpe_multi* mm, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                        const double* weights, double* cost, double* grad) {
    return gpe_multi_bank_cost_ex(mm, testing, N, obs, obs_ld, weights, cost, grad, nullptr);
}

int gpe_multi_bank_forward_cost_ex(gpe_multi* mm, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                                   const double* weights, double* cost, double* grad, double* hess) {
    NvtxRange nvtx_range("gpe_multi_bank_forward_cost");
    return multi_bank_cost_call(mm, testing, N, obs, obs_ld, weights, 0, cost, grad, hess, true);
}

int gpe_multi_bank_forward_cost(gpe_multi* mm, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                                const double* weights, double* cost, double* grad) {
    return gpe_multi_bank_forward_cost_ex(mm, testing, N, obs, obs_ld, weights, cost, grad, nullptr);
}

int gpe_multi_bank_solve(gpe_multi* mm, const double* x0, int64_t N, const double* obs, int64_t obs_ld, const double* weights,
                         const gpe_solve_opts* opts, double* x, double* cost, double* grad, double* hess, double* cov,
                         int32_t* info, unsigned flags) {
    return gpe_multi_bank_solve_pw(mm, x0, N, obs, obs_ld, weights, 0, opts, x, cost, grad, hess, cov, info, flags);
}

int gpe_multi_bank_solve_pw(gpe_multi* mm, const double* x0, int64_t N, const double* obs, int64_t obs_ld, const double* weights,
                            int64_t weights_ld, const gpe_solve_opts* opts, double* x, double* cost, double* grad, double* hess,
                            double* cov, int32_t* info, unsigned flags) {
    NvtxRange nvtx_range("gpe_multi_bank_solve");
    if (!mm || mm->banks.empty()) return fail(GPE_ERR_INVALID, "handle is NULL or not a bank handle");
    gpe_bank* b0 = mm->banks[0];
    const bool spectra = flags & GPE_SOLVE_SPECTRA;
    gpe_solve_opts o;
    int rc = solve_check(b0, N, x0, obs, obs_ld, opts, x, info, flags, true, nullptr, &o);
    if (rc == GPE_OK) rc = weights_check(weights, weights_ld, spectra ? b0->W : b0->E, spectra, true);
    if (rc || N == 0) return rc;
    const SolveIo s = solve_io(b0->D, spectra ? b0->W : b0->E, x0, obs, obs_ld, o, x, cost, grad, hess, cov, info, weights,
                               weights_ld);
    return fan_out(mm, mm->banks, b0->models[0]->sms, s.io, N, -1, [&](gpe_bank* b, const SharedCall* shared) {
        return bank_solve_stream(b, spectra, N, obs, obs_ld, weights, o, s, shared);
    });
}

int gpe_multi_bank_solve_series(gpe_multi* mm, int64_t S, int64_t T, const double* x0, const double* obs, int64_t obs_ld,
                                const double* weights, int64_t weights_ld, const gpe_solve_opts* opts, const double* smooth_prec,
                                const double* coupling, double* x, double* cost, double* grad, double* hess, double* cov,
                                int32_t* info, unsigned flags) {
    NvtxRange nvtx_range("gpe_multi_bank_solve_series");
    if (!mm || mm->banks.empty()) return fail(GPE_ERR_INVALID, "handle is NULL or not a bank handle");
    gpe_bank* b0 = mm->banks[0];
    const bool spectra = flags & GPE_SOLVE_SPECTRA;
    int rc = series_check(b0, S, T, smooth_prec, coupling, true, nullptr);
    gpe_solve_opts o;
    if (rc == GPE_OK) rc = solve_check(b0, S * T, x0, obs, obs_ld, opts, x, info, flags, true, nullptr, &o);
    if (rc == GPE_OK) rc = weights_check(weights, weights_ld, spectra ? b0->W : b0->E, spectra, true);
    if (rc || S == 0) return rc;
    const SolveIo s = solve_io(b0->D, spectra ? b0->W : b0->E, x0, obs, obs_ld, o, x, cost, grad, hess, cov, info, weights,
                               weights_ld, T);
    const LmSeries sp{(int)T, coupling, smooth_prec, nullptr};
    return fan_out(mm, mm->banks, b0->models[0]->sms, s.io, S, -1, [&](gpe_bank* b, const SharedCall* shared) {
        return bank_solve_stream(b, spectra, S, obs, obs_ld, weights, o, s, shared, &sp);
    });
}

int gpe_multi_bank_search(gpe_multi* mm, const double* cand, int64_t K, const double* obs, int64_t N, int64_t obs_ld,
                          const double* weights, int k, int64_t* idx, double* cost, unsigned flags) {
    return gpe_multi_bank_search_pw(mm, cand, K, obs, N, obs_ld, weights, 0, k, idx, cost, flags);
}

int gpe_multi_bank_search_pw(gpe_multi* mm, const double* cand, int64_t K, const double* obs, int64_t N, int64_t obs_ld,
                             const double* weights, int64_t weights_ld, int k, int64_t* idx, double* cost, unsigned flags) {
    NvtxRange nvtx_range("gpe_multi_bank_search");
    if (!mm || mm->banks.empty()) return fail(GPE_ERR_INVALID, "handle is NULL or not a bank handle");
    gpe_bank* b0 = mm->banks[0];
    const bool spectra = flags & GPE_SOLVE_SPECTRA;
    int rc = search_check(b0, cand, K, obs, N, obs_ld, k, idx, cost, flags, true, weights, weights_ld);
    if (rc || N == 0) return rc;
    const CallIo io = search_io(spectra ? b0->W : b0->E, obs, obs_ld, k, idx, cost, weights, weights_ld);
    // every device builds its own, identical candidate table
    return fan_out(mm, mm->banks, b0->models[0]->sms, io, N, -1, [&](gpe_bank* b, const SharedCall* shared) {
        return bank_search_stream(b, spectra, cand, K, obs, N, obs_ld, weights, k, io, shared, weights_ld);
    });
}

}  // extern "C"
