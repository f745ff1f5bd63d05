// Host-resident callers: the chunked, overlapped H2D -> kernels -> D2H pipeline shared by every entry point that takes
// GPE_HOST_PTRS (single GP, FP32, banks, bank cost, bank forward) and by the one-call multi-device fan-out.
//
// Replaces the Python chunk loop of GaussianProcess.gpu_predict / get_gpu_block (reference
// gp_emulator/GaussianProcess.py:253-323: slice, cast, predict_wrap per block, np.append), which the reference's own
// report names as 34 % of the GPU path's wall time (doc/report.md:70).
//
//   pinned caller buffers   : DMA'd directly, two slots;
//   pageable caller buffers : staged through page-locked slot buffers -- inputs and outputs independently, so a caller
//                             with pageable inputs and page-locked result arrays only pays for the copy-in.  The caller's
//                             thread stages inputs and enqueues (copy-in -> H2D -> kernels -> D2H -> event), a second
//                             thread waits for each chunk's event and copies its results out, both through the CopyPool;
//                             three slots keep the GPU busy while either side is late;
//   tiny calls              : the kernels run directly on the page-locked staging buffers (mapped, UVA): one launch and
//                             one synchronisation, no copy calls.
// Chunks come from a ChunkSource -- an atomic cursor over [0, N) -- so that several devices can pull from ONE call's
// point range (gpe_multi_*): a device behind a slower PCIe link simply takes fewer chunks.  Test points are independent
// (GaussianProcess.py:228-249) and the kernels' results do not depend on a point's position in a launch, so any split
// reproduces the single-device result bit for bit.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <thread>
#include <vector>

#include "../../include/gpemu.h"
#include "host_common.h"

namespace gpe {

#define GPE_CUDA_TRY(expr)                                                                                        \
    do {                                                                                                          \
        cudaError_t _e = (expr);                                                                                  \
        if (_e != cudaSuccess)                                                                                    \
            return ::gpe::set_error(GPE_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

constexpr int64_t kPipeChunk = 1 << 18;   // points per host-streaming chunk (single GP: 20 MB in, 25 MB out)
constexpr int64_t kZeroCopyMax = 16384;   // host calls of up to this many points run on mapped page-locked buffers
                                          // (tools/zero_copy_probe.py: 1000 points 71 -> 58 us, 16000 points 470 -> 300 us)
constexpr size_t kSlotOutBytes = (size_t)512 << 20;   // cap of one slot's result buffer: bounds chunks of wide outputs
                                                      // (bank Hessians: 57 KB per point, spectra: 17 KB per point)
constexpr size_t kSlotInBytes = (size_t)1 << 30;      // cap of one slot's input buffer: bounds chunks of wide inputs (observed
                                                      // spectra: 17 KB per point).  Binds only above 512 doubles per point
                                                      // (kPipeChunk x 4 KB): test points (D <= GPE_MAX_INPUTS = 256) never
                                                      // reach it, band observations only where D + E > 512
constexpr int kMaxIo = 8;

struct Slot {
    cudaStream_t st = nullptr;
    cudaEvent_t done = nullptr;
    void* d_in = nullptr;
    void* d_out = nullptr;
    void* h_in = nullptr;    // pinned staging (pageable callers only)
    void* h_out = nullptr;
    size_t d_in_cap = 0, d_out_cap = 0, h_in_cap = 0, h_out_cap = 0;
    int64_t pend_n0 = 0, pend_n = 0;   // chunk whose results wait in h_out (staged path)
};

inline void free_slot(Slot& s) {
    if (s.d_in) cudaFree(s.d_in);
    if (s.d_out) cudaFree(s.d_out);
    if (s.h_in) cudaFreeHost(s.h_in);
    if (s.h_out) cudaFreeHost(s.h_out);
    if (s.done) cudaEventDestroy(s.done);
    if (s.st) cudaStreamDestroy(s.st);
    s = Slot();
}

inline bool is_pinned_or_null(const void* p) {
    if (p == nullptr) return true;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

inline int ensure_buf(void** ptr, size_t* cap, size_t need, bool host) {
    if (*cap >= need) return GPE_OK;
    if (*ptr) {
        if (host) cudaFreeHost(*ptr); else cudaFree(*ptr);
        *ptr = nullptr; *cap = 0;
    }
    if (host) GPE_CUDA_TRY(cudaMallocHost(ptr, need));
    else GPE_CUDA_TRY(cudaMalloc(ptr, need));
    *cap = need;
    return GPE_OK;
}

// Staging copies for pageable callers.  One core moves ~14 GB/s on the GPU boxes, eight ~50 GB/s, and the PCIe link
// 55 GB/s each way, so copies of 1 MB and more are split into >= 256 KB pieces over a small persistent pool (created on
// first use; the submitting thread takes a share of the pieces itself).  Several threads may submit at once: the staged
// pipeline copies results out on its own thread while the caller's thread stages the next inputs.
class CopyPool {
public:
    static CopyPool& get() {
        static CopyPool pool;
        return pool;
    }
    void copy(void* dst, const void* src, size_t bytes) {
        constexpr size_t kPiece = 256u << 10;   // waking a worker costs tens of microseconds: not worth it below 1 MB
        const size_t want = bytes >= 4 * kPiece ? bytes / kPiece : 1;
        const unsigned np = (unsigned)std::min<size_t>(workers_.size() + 1, std::max<size_t>(want, 1));
        if (np <= 1) {
            memcpy(dst, src, bytes);
            return;
        }
        const size_t part = (bytes / np + 63) & ~(size_t)63;
        Batch batch;
        unsigned queued = 0;
        {
            std::lock_guard<std::mutex> lk(mu_);
            for (unsigned i = 1; i < np; ++i) {
                const size_t off = (size_t)i * part;
                if (off >= bytes) break;
                q_.push_back(Task{(char*)dst + off, (const char*)src + off, std::min(part, bytes - off), &batch});
                ++queued;
            }
            batch.remaining = (int)queued;
        }
        cv_.notify_all();
        memcpy(dst, src, std::min(part, bytes));
        std::unique_lock<std::mutex> lk(mu_);
        done_cv_.wait(lk, [&] { return batch.remaining == 0; });
    }

private:
    struct Batch { int remaining = 0; };
    struct Task { char* dst; const char* src; size_t len; Batch* batch; };
    CopyPool() {
        const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
        const unsigned n = std::min(7u, std::max(1u, hw / 2) - (hw >= 4 ? 1u : 0u));
        for (unsigned i = 0; i < n; ++i) workers_.emplace_back([this] { run(); });
    }
    ~CopyPool() {
        {
            std::lock_guard<std::mutex> lk(mu_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto& t : workers_) t.join();
    }
    void run() {
        std::unique_lock<std::mutex> lk(mu_);
        for (;;) {
            cv_.wait(lk, [&] { return stop_ || !q_.empty(); });
            if (stop_) return;
            Task t = q_.front();
            q_.pop_front();
            lk.unlock();
            memcpy(t.dst, t.src, t.len);
            lk.lock();
            if (--t.batch->remaining == 0) done_cv_.notify_all();
        }
    }
    std::vector<std::thread> workers_;
    std::deque<Task> q_;
    std::mutex mu_;
    std::condition_variable cv_, done_cv_;
    bool stop_ = false;
};

inline void par_memcpy(void* dst, const void* src, size_t bytes) { CopyPool::get().copy(dst, src, bytes); }

// One streamed array: `width` elements per test point.  Inputs: host != NULL.  Outputs: host == NULL marks a
// device-only intermediate of the chunk (e.g. the PC means a back-projection consumes) that is never copied out.
struct IoSpec {
    void* host;
    int64_t width;
};

struct ChunkSource {
    std::atomic<int64_t>* cursor;
    int64_t N, CH;
    bool take(int64_t* n0, int64_t* n) {
        const int64_t s = cursor->fetch_add(CH, std::memory_order_relaxed);
        if (s >= N) return false;
        *n0 = s;
        *n = std::min(CH, N - s);
        return true;
    }
};

// NVLink relay of one device's host traffic through a partner device's PCIe link (gpe_multi_*: on some boxes half of
// the GPUs sit behind a slower PCIe path, profiles/r02_pcie_probe8_*.txt).  Buffers, streams and the in / done events
// live on the partner; ev_out on the device itself.  Two slots, matching the direct path.
struct Relay {
    int partner = -1;
    cudaStream_t st[2] = {nullptr, nullptr};
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr}, done[2] = {nullptr, nullptr};
    void* r_in[2] = {nullptr, nullptr};
    void* r_out[2] = {nullptr, nullptr};
    size_t in_cap[2] = {0, 0}, out_cap[2] = {0, 0};
};

struct StreamPlan {
    bool in_direct = false, out_direct = false, zero_copy = false;
    int64_t CH = 1;
    int nslots = 2;
};

inline size_t io_bytes(const IoSpec* io, int nio, int64_t n, size_t ES, bool external_only) {
    size_t b = 0;
    for (int i = 0; i < nio; ++i)
        if (!external_only || io[i].host) b += ((size_t)n * io[i].width * ES + 255) & ~(size_t)255;
    return b;
}

// Decide how one call of N points is streamed.  `wave` = points of one wave of tiles on one device (64 x #SM);
// n_devices > 1: the chunks are shared by that many pipelines pulling from one cursor.
inline StreamPlan plan_stream(const IoSpec* ins, int nin, const IoSpec* outs, int nout, int64_t N, size_t ES, int64_t wave,
                              int n_devices, bool allow_zero_copy) {
    StreamPlan pl;
    // inputs and outputs are staged independently: page-locked caller memory is DMA'd directly on either side
    // (a pointer query on pageable memory costs ~10 us: a small call with pageable inputs does not ask about its
    // outputs -- staging a few KB is cheaper than finding out)
    pl.in_direct = true;
    for (int i = 0; i < nin; ++i) pl.in_direct = pl.in_direct && is_pinned_or_null(ins[i].host);
    const bool tiny = N <= 3 * wave;
    pl.out_direct = pl.in_direct || !tiny;
    for (int i = 0; i < nout && pl.out_direct; ++i) pl.out_direct = is_pinned_or_null(outs[i].host);
    int64_t per_in = 0, per_out = 0;
    for (int i = 0; i < nin; ++i) per_in += ins[i].width;
    for (int i = 0; i < nout; ++i) per_out += outs[i].width;
    // wide outputs (inputs) bound the chunk through the slot's result (input) buffer, in whole waves where that leaves at
    // least one
    int64_t cap = kPipeChunk;
    size_t slot_bytes = kSlotOutBytes;
    if (const char* e = getenv("GPE_SLOT_OUT_BYTES")) slot_bytes = (size_t)atoll(e);   // dev aid: force chunk seams in tests
    if (per_out > 0) cap = std::min<int64_t>(cap, (int64_t)(slot_bytes / ((size_t)per_out * ES)));
    if (per_in > 0) cap = std::min<int64_t>(cap, (int64_t)(kSlotInBytes / ((size_t)per_in * ES)));
    if (cap >= wave) cap = cap / wave * wave;
    cap = std::max<int64_t>(cap, 1);
    const bool direct = pl.in_direct && pl.out_direct;
    if (direct && n_devices == 1) {
        pl.CH = std::min<int64_t>(cap, std::max<int64_t>(N, 1));
    } else {
        // about a quarter of each pipeline's share, whole waves, so that mid-sized calls overlap (and balance) too
        const int64_t share = (N + n_devices - 1) / n_devices;
        pl.CH = std::min<int64_t>(cap, std::max<int64_t>(std::min<int64_t>(2 * wave, cap), ((share + 3) / 4 + wave - 1) / wave * wave));
        if (n_devices == 1 && N <= 3 * wave && N <= cap) pl.CH = std::max<int64_t>(N, 1);   // too small to be worth a second thread
    }
    pl.nslots = direct ? 2 : 3;
    static const bool no_zero_copy = getenv("GPE_NO_ZERO_COPY") != nullptr;   // dev aid: time the copy-based small path
    static const int64_t zc_max = getenv("GPE_ZERO_COPY_MAX") ? atoll(getenv("GPE_ZERO_COPY_MAX")) : kZeroCopyMax;   // dev aid
    // (results are written over PCIe by the kernels themselves: only worth it while they are small)
    pl.zero_copy = allow_zero_copy && n_devices == 1 && N <= zc_max && N <= pl.CH && !pl.in_direct && !pl.out_direct &&
                   !no_zero_copy && io_bytes(outs, nout, N, ES, true) <= ((size_t)2 << 20);
    return pl;
}

// Grow the slots' buffers for the plan (idempotent; called under the owner's host mutex).
inline int prepare_slots(Slot* slots, const StreamPlan& pl, const IoSpec* ins, int nin, const IoSpec* outs, int nout, size_t ES) {
    const size_t in_b = std::max<size_t>(io_bytes(ins, nin, pl.CH, ES, false), 256);
    const size_t out_b = std::max<size_t>(io_bytes(outs, nout, pl.CH, ES, false), 256);
    const size_t out_ext = std::max<size_t>(io_bytes(outs, nout, pl.CH, ES, true), 256);
    for (int i = 0; i < pl.nslots; ++i) {
        Slot& s = slots[i];
        if (!s.st) GPE_CUDA_TRY(cudaStreamCreateWithFlags(&s.st, cudaStreamNonBlocking));
        if (!s.done) GPE_CUDA_TRY(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
        int rc = GPE_OK;
        if (!pl.zero_copy) {
            rc = ensure_buf(&s.d_in, &s.d_in_cap, in_b, false);
            if (rc) return rc;
        }
        // (the zero-copy path keeps device-only intermediates in d_out and external results in h_out)
        rc = ensure_buf(&s.d_out, &s.d_out_cap, out_b, false);
        if (rc) return rc;
        if (!pl.in_direct) {
            rc = ensure_buf(&s.h_in, &s.h_in_cap, in_b, true);
            if (rc) return rc;
        }
        if (!pl.out_direct) {
            rc = ensure_buf(&s.h_out, &s.h_out_cap, out_ext, true);
            if (rc) return rc;
        }
    }
    return GPE_OK;
}

// Run one pipeline (one device) until the chunk source is exhausted.
//   launch(n0, n, d_ins, d_outs, stream) enqueues the kernels of chunk [n0, n0 + n): d_ins[i] / d_outs[i] are the
//   chunk-local device arrays ((n, width) each, 256-byte aligned; external outputs first, then the intermediates).
template <typename Launch>
int stream_host(Slot* slots, int device, const StreamPlan& pl, ChunkSource src, size_t ES, const IoSpec* ins, int nin,
                const IoSpec* outs, int nout, Launch launch, const Relay* relay = nullptr) {
    if (relay && !(pl.in_direct && pl.out_direct)) relay = nullptr;   // the staged path copies through its own slots
    if (nin > kMaxIo || nout > kMaxIo) return set_error(GPE_ERR_INVALID, "too many streamed arrays");
    // order of the chunk-local output arrays: external ones first (one contiguous D2H in the staged path)
    int order[kMaxIo], next = 0;
    for (int i = 0; i < nout; ++i) if (outs[i].host) order[next++] = i;
    const int n_ext = next;
    for (int i = 0; i < nout; ++i) if (!outs[i].host) order[next++] = i;
    auto carve = [&](void* base, void* base_int, const IoSpec* io, int nio, const int* ord, int n_first, int64_t n, void** ptrs) {
        // arrays ord[0 .. n_first) from `base`, the rest from `base_int` (continuing after them when both are one buffer)
        char* p = (char*)base;
        for (int k = 0; k < nio; ++k) {
            if (k == n_first && base_int != nullptr) p = (char*)base_int;
            const int i = ord ? ord[k] : k;
            ptrs[i] = p;
            p += ((size_t)n * io[i].width * ES + 255) & ~(size_t)255;
        }
    };
    auto h2d = [&](Slot& s, void* const* d_ins, const void* stage, int64_t n0, int64_t n) -> int {
        const char* sp = (const char*)stage;
        for (int i = 0; i < nin; ++i) {
            const size_t bytes = (size_t)n * ins[i].width * ES;
            const void* from = stage ? (const void*)sp : (const void*)((const char*)ins[i].host + (size_t)n0 * ins[i].width * ES);
            GPE_CUDA_TRY(cudaMemcpyAsync(d_ins[i], from, bytes, cudaMemcpyHostToDevice, s.st));
            sp += (bytes + 255) & ~(size_t)255;
        }
        return GPE_OK;
    };
    auto d2h_direct = [&](Slot& s, void* const* d_outs, int64_t n0, int64_t n) -> int {
        for (int i = 0; i < nout; ++i)
            if (outs[i].host)
                GPE_CUDA_TRY(cudaMemcpyAsync((char*)outs[i].host + (size_t)n0 * outs[i].width * ES, d_outs[i],
                                             (size_t)n * outs[i].width * ES, cudaMemcpyDeviceToHost, s.st));
        return GPE_OK;
    };
    void *d_ins[kMaxIo], *d_outs[kMaxIo];
    int64_t n0 = 0, n = 0;

    if (pl.in_direct && pl.out_direct) {
        // At most two chunks in flight per pipeline: a slot takes its next chunk only when its previous one has finished,
        // so that with several pipelines on one cursor a chunk goes to the device that is ready for it (taking chunks at
        // enqueue speed would hand the whole call to the first thread).
        int which = 0;
        bool used[2] = {false, false};
        for (;;) {
            Slot& s = slots[which];
            cudaEvent_t done = relay ? relay->done[which] : s.done;
            if (used[which]) GPE_CUDA_TRY(cudaEventSynchronize(done));
            if (!src.take(&n0, &n)) break;
            used[which] = true;
            carve(s.d_in, nullptr, ins, nin, nullptr, nin, n, d_ins);
            carve(s.d_out, nullptr, outs, nout, order, nout, n, d_outs);
            int rc;
            if (!relay) {
                rc = h2d(s, d_ins, nullptr, n0, n);
                if (rc) return rc;
                rc = launch(n0, n, d_ins, d_outs, s.st);
                if (rc) return rc;
                rc = d2h_direct(s, d_outs, n0, n);
                if (rc) return rc;
                GPE_CUDA_TRY(cudaEventRecord(s.done, s.st));
            } else {
                // Host traffic of this device rides the partner's PCIe link: host -> partner (H2D on the partner's stream)
                // -> NVLink peer copy -> kernels here -> NVLink peer copy -> partner -> host.
                void *r_ins[kMaxIo], *r_outs[kMaxIo];
                carve(relay->r_in[which], nullptr, ins, nin, nullptr, nin, n, r_ins);
                carve(relay->r_out[which], nullptr, outs, nout, order, nout, n, r_outs);
                cudaStream_t rst = relay->st[which];
                GPE_CUDA_TRY(cudaSetDevice(relay->partner));
                for (int i = 0; i < nin; ++i)
                    GPE_CUDA_TRY(cudaMemcpyAsync(r_ins[i], (const char*)ins[i].host + (size_t)n0 * ins[i].width * ES,
                                                 (size_t)n * ins[i].width * ES, cudaMemcpyHostToDevice, rst));
                GPE_CUDA_TRY(cudaEventRecord(relay->ev_in[which], rst));
                GPE_CUDA_TRY(cudaSetDevice(device));
                GPE_CUDA_TRY(cudaStreamWaitEvent(s.st, relay->ev_in[which], 0));
                GPE_CUDA_TRY(cudaMemcpyPeerAsync(s.d_in, device, relay->r_in[which], relay->partner, io_bytes(ins, nin, n, ES, false), s.st));
                rc = launch(n0, n, d_ins, d_outs, s.st);
                if (rc) return rc;
                GPE_CUDA_TRY(cudaMemcpyPeerAsync(relay->r_out[which], relay->partner, s.d_out, device, io_bytes(outs, nout, n, ES, true), s.st));
                GPE_CUDA_TRY(cudaEventRecord(relay->ev_out[which], s.st));
                GPE_CUDA_TRY(cudaSetDevice(relay->partner));
                GPE_CUDA_TRY(cudaStreamWaitEvent(rst, relay->ev_out[which], 0));
                for (int i = 0; i < nout; ++i)
                    if (outs[i].host)
                        GPE_CUDA_TRY(cudaMemcpyAsync((char*)outs[i].host + (size_t)n0 * outs[i].width * ES, r_outs[i],
                                                     (size_t)n * outs[i].width * ES, cudaMemcpyDeviceToHost, rst));
                GPE_CUDA_TRY(cudaEventRecord(relay->done[which], rst));
                GPE_CUDA_TRY(cudaSetDevice(device));
            }
            which ^= 1;
        }
        for (int i = 0; i < 2; ++i)
            if (used[i]) GPE_CUDA_TRY(cudaEventSynchronize(relay ? relay->done[i] : slots[i].done));
        return GPE_OK;
    }

    // ---- staged path (inputs and / or outputs in pageable memory) -------------------------------------------
    static const bool pipe_trace = getenv("GPE_PIPE_TRACE") != nullptr;   // dev aid: host-side time split of a call
    double t_wait = 0, t_out = 0, t_in = 0, t_block = 0;
    int64_t chunks_done = 0;
    auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    auto scatter_out = [&](const void* stage, int64_t c0, int64_t cn) {   // staged results -> the caller's arrays
        const char* sp = (const char*)stage;
        for (int k = 0; k < n_ext; ++k) {
            const int i = order[k];
            const size_t bytes = (size_t)cn * outs[i].width * ES;
            par_memcpy((char*)outs[i].host + (size_t)c0 * outs[i].width * ES, sp, bytes);
            sp += (bytes + 255) & ~(size_t)255;
        }
    };
    auto gather_in = [&](void* stage, int64_t c0, int64_t cn, bool parallel) {
        char* sp = (char*)stage;
        for (int i = 0; i < nin; ++i) {
            const size_t bytes = (size_t)cn * ins[i].width * ES;
            const void* from = (const char*)ins[i].host + (size_t)c0 * ins[i].width * ES;
            if (parallel) par_memcpy(sp, from, bytes); else memcpy(sp, from, bytes);
            sp += (bytes + 255) & ~(size_t)255;
        }
    };
    auto copy_out = [&](Slot& s) -> cudaError_t {   // wait for the slot's chunk, then scatter its results to the caller
        double t0 = now();
        cudaError_t e = cudaEventSynchronize(s.done);
        if (e != cudaSuccess) return e;
        t_wait += now() - t0; t0 = now();
        if (pl.out_direct) return cudaSuccess;          // the D2H copies went straight into the caller's arrays
        scatter_out(s.h_out, s.pend_n0, s.pend_n);
        t_out += now() - t0;
        return cudaSuccess;
    };
    auto stage_in = [&](Slot& s, int64_t c0, int64_t cn) -> int {   // copy-in + enqueue of one chunk on the slot
        void *di[kMaxIo], *dout[kMaxIo];
        carve(s.d_in, nullptr, ins, nin, nullptr, nin, cn, di);
        carve(s.d_out, nullptr, outs, nout, order, nout, cn, dout);
        int rc;
        if (pl.in_direct) {
            rc = h2d(s, di, nullptr, c0, cn);
        } else {
            double t0 = now();
            gather_in(s.h_in, c0, cn, true);
            t_in += now() - t0;
            rc = h2d(s, di, s.h_in, c0, cn);
        }
        if (rc) return rc;
        rc = launch(c0, cn, di, dout, s.st);
        if (rc) return rc;
        if (pl.out_direct) {
            rc = d2h_direct(s, dout, c0, cn);
            if (rc) return rc;
        } else if (n_ext > 0) {
            GPE_CUDA_TRY(cudaMemcpyAsync(s.h_out, s.d_out, io_bytes(outs, nout, cn, ES, true), cudaMemcpyDeviceToHost, s.st));
        }
        GPE_CUDA_TRY(cudaEventRecord(s.done, s.st));
        s.pend_n0 = c0; s.pend_n = cn;
        return GPE_OK;
    };
    int rc = GPE_OK;
    if (pl.zero_copy) {
        // Small calls (the reference is typically called with ONE point): the two cudaMemcpyAsync of the staged
        // path cost more than the kernel.  The staging buffers are page-locked, hence mapped into the device's address
        // space (UVA): the kernels read the test rows from and write the results to host memory directly -- one launch
        // and one synchronisation instead of copy, launch, copy, synchronise.
        if (!src.take(&n0, &n)) return GPE_OK;
        Slot& s = slots[0];
        double t0 = now();
        gather_in(s.h_in, n0, n, false);
        t_in += now() - t0;
        carve(s.h_in, nullptr, ins, nin, nullptr, nin, n, d_ins);
        carve(s.h_out, s.d_out, outs, nout, order, n_ext, n, d_outs);
        rc = launch(n0, n, d_ins, d_outs, s.st);
        if (rc) return rc;
        t0 = now();
        GPE_CUDA_TRY(cudaStreamSynchronize(s.st));
        t_wait += now() - t0; t0 = now();
        const char* sp = (const char*)s.h_out;
        for (int k = 0; k < n_ext; ++k) {
            const int i = order[k];
            const size_t bytes = (size_t)n * outs[i].width * ES;
            memcpy((char*)outs[i].host + (size_t)n0 * outs[i].width * ES, sp, bytes);
            sp += (bytes + 255) & ~(size_t)255;
        }
        t_out += now() - t0;
        chunks_done = 1;
    } else if (pl.out_direct) {
        // only the inputs are staged: no second thread, a slot is reused once its previous chunk has finished
        int64_t c = 0;
        for (; src.take(&n0, &n); ++c) {
            Slot& s = slots[c % 3];
            if (c >= 3) {
                const double t0 = now();
                GPE_CUDA_TRY(cudaEventSynchronize(s.done));
                t_block += now() - t0;
            }
            rc = stage_in(s, n0, n);
            if (rc) { cudaDeviceSynchronize(); return rc; }
        }
        for (int i = 0; i < 3 && i < c; ++i) GPE_CUDA_TRY(cudaStreamSynchronize(slots[i].st));
        chunks_done = c;
    } else {
        // chunk c of this pipeline lives in slot c % 3.  `staged` / `drained` count chunks handed to / finished by the
        // output thread; `finished` says the source is exhausted.
        std::mutex mx;
        std::condition_variable cv;
        int64_t staged = 0, drained = 0;
        bool abort = false, finished = false;
        cudaError_t out_err = cudaSuccess;
        std::thread out_thread;
        bool have_thread = false;
        auto out_loop = [&] {
            cudaSetDevice(device);
            for (int64_t c = 0;; ++c) {
                {
                    std::unique_lock<std::mutex> lk(mx);
                    cv.wait(lk, [&] { return staged > c || abort || finished; });
                    if (staged <= c) return;
                }
                const cudaError_t e = copy_out(slots[c % 3]);
                std::lock_guard<std::mutex> lk(mx);
                if (e != cudaSuccess) { out_err = e; abort = true; cv.notify_all(); return; }
                drained = c + 1;
                cv.notify_all();
            }
        };
        int64_t c = 0;
        for (; rc == GPE_OK && src.take(&n0, &n); ++c) {
            if (c == 1 && !have_thread) { out_thread = std::thread(out_loop); have_thread = true; }
            if (have_thread) {
                const double t0 = now();
                std::unique_lock<std::mutex> lk(mx);
                cv.wait(lk, [&] { return drained + 3 > c || abort; });   // the slot's previous chunk has left it
                if (abort) break;
                t_block += now() - t0;
            }
            rc = stage_in(slots[c % 3], n0, n);
            std::lock_guard<std::mutex> lk(mx);
            if (rc == GPE_OK) staged = c + 1; else abort = true;
            cv.notify_all();
        }
        {
            std::lock_guard<std::mutex> lk(mx);
            finished = true;
            cv.notify_all();
        }
        if (have_thread) {
            out_thread.join();
        } else if (rc == GPE_OK && staged == 1) {     // a single chunk: no second thread
            const cudaError_t e = copy_out(slots[0]);
            if (e != cudaSuccess) out_err = e;
        }
        if (rc) {                     // stage_in failed: the error text is already set on this thread
            cudaDeviceSynchronize();
            return rc;
        }
        if (out_err != cudaSuccess) return set_error(GPE_ERR_CUDA, "result copy-out failed: %s", cudaGetErrorString(out_err));
        chunks_done = c;
    }
    if (pipe_trace)
        fprintf(stderr, "[gpemu pipe] device %d: %lld chunks of <= %lld points (in %s, out %s%s): out-thread wait %.3f ms, copy-out %.3f ms | "
                        "copy-in %.3f ms, caller blocked on a slot %.3f ms\n",
                device, (long long)chunks_done, (long long)pl.CH, pl.in_direct ? "direct" : "staged",
                pl.out_direct ? "direct" : "staged", pl.zero_copy ? ", mapped" : "", t_wait * 1e3, t_out * 1e3, t_in * 1e3, t_block * 1e3);
    return GPE_OK;
}

}  // namespace gpe
