// PCIe / host-memory fabric probe for the host-resident (e2e) path: ONE process, one thread per GPU, every GPU copying
// at the same time.  Answers (VERDICT r01 "what's weak" #2): is the D2H ceiling per GPU or shared, does it move with
// hugepage-backed page-locked memory, do time-multiplexed H2D / D2H phases beat concurrent copies, does copy size matter.
//   nvcc -O2 -std=c++17 -o build/pcie_probe tools/pcie_probe.cu -lpthread     ;   build/pcie_probe [seconds-per-case]
#include <cuda_runtime.h>
#include <pthread.h>
#include <sched.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <atomic>
#include <chrono>
#include <string>
#include <thread>
#include <vector>

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "%s: %s (line %d)\n", #x, cudaGetErrorString(e_), __LINE__); exit(1); } } while (0)

static double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

enum BufKind { PINNED, PINNED_WC, THP_REG, HUGETLB_REG };
static const char* kind_name[] = {"cudaHostAlloc", "cudaHostAlloc(WC)", "mmap+THP+register", "mmap(HUGETLB)+register"};

static void* host_buf(BufKind k, size_t bytes) {
    void* p = nullptr;
    if (k == PINNED) { CK(cudaHostAlloc(&p, bytes, cudaHostAllocPortable)); memset(p, 1, bytes); return p; }
    if (k == PINNED_WC) { CK(cudaHostAlloc(&p, bytes, cudaHostAllocPortable | cudaHostAllocWriteCombined)); memset(p, 1, bytes); return p; }
    int flags = MAP_PRIVATE | MAP_ANONYMOUS | (k == HUGETLB_REG ? MAP_HUGETLB : 0);
    p = mmap(nullptr, bytes, PROT_READ | PROT_WRITE, flags, -1, 0);
    if (p == MAP_FAILED) return nullptr;
    if (k == THP_REG) madvise(p, bytes, MADV_HUGEPAGE);
    memset(p, 1, bytes);
    if (cudaHostRegister(p, bytes, cudaHostRegisterPortable) != cudaSuccess) { cudaGetLastError(); munmap(p, bytes); return nullptr; }
    return p;
}

static std::vector<int> local_cpus(int dev) {
    char bdf[32]; std::vector<int> cpus;
    if (cudaDeviceGetPCIBusId(bdf, sizeof(bdf), dev) != cudaSuccess) return cpus;
    for (char* c = bdf; *c; ++c) *c = (char)tolower(*c);
    std::string path = std::string("/sys/bus/pci/devices/") + bdf + "/local_cpulist";
    FILE* f = fopen(path.c_str(), "r");
    if (!f) return cpus;
    char line[4096];
    if (fgets(line, sizeof(line), f)) {
        for (char* tok = strtok(line, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
            int a, b; if (sscanf(tok, "%d-%d", &a, &b) == 2) { for (int i = a; i <= b; ++i) cpus.push_back(i); } else if (sscanf(tok, "%d", &a) == 1) cpus.push_back(a);
        }
    }
    fclose(f);
    return cpus;
}

struct Dev { int id; void *h_in, *h_out, *d_in, *d_out; cudaStream_t s_in, s_out; };

// mode: 1 = H2D only, 2 = D2H only, 3 = both concurrently (two streams), 4 = alternating phases (H2D chunk, then D2H chunk, one stream)
static std::vector<double> run_case(std::vector<Dev>& devs, const std::vector<int>& active, int mode_all, size_t chunk, size_t total, double secs,
                                    const std::vector<int>* modes = nullptr) {
    std::vector<double> rate(devs.size(), 0.0);
    std::atomic<int> ready{0}; std::atomic<bool> go{false};
    std::vector<std::thread> th;
    for (int g : active) th.emplace_back([&, g] {
        Dev& d = devs[g];
        const int mode = modes ? (*modes)[g] : mode_all;
        CK(cudaSetDevice(d.id));
        ready++; while (!go.load()) {}
        const double t0 = now(); size_t moved = 0; size_t off = 0;
        while (now() - t0 < secs) {
            for (int rep = 0; rep < 4; ++rep) {
                if (off + chunk > total) off = 0;
                if (mode & 1) CK(cudaMemcpyAsync((char*)d.d_in + off, (char*)d.h_in + off, chunk, cudaMemcpyHostToDevice, d.s_in));
                if (mode == 4) CK(cudaMemcpyAsync((char*)d.h_out + off, (char*)d.d_out + off, chunk, cudaMemcpyDeviceToHost, d.s_in));
                else if (mode & 2) CK(cudaMemcpyAsync((char*)d.h_out + off, (char*)d.d_out + off, chunk, cudaMemcpyDeviceToHost, d.s_out));
                off += chunk; moved += chunk;
            }
            CK(cudaStreamSynchronize(d.s_in)); CK(cudaStreamSynchronize(d.s_out));
        }
        rate[g] = moved / (now() - t0) / 1e9;   // per direction
    });
    while (ready.load() < (int)active.size()) {}
    go = true;
    for (auto& t : th) t.join();
    return rate;
}

int main(int argc, char** argv) {
    const double secs = argc > 1 ? atof(argv[1]) : 0.6;
    int G = 0; CK(cudaGetDeviceCount(&G));
    const size_t total = (size_t)512 << 20;
    printf("devices: %d\n", G);
    {   // hugepage availability
        FILE* f = fopen("/proc/meminfo", "r"); char line[256];
        while (f && fgets(line, sizeof(line), f)) if (strstr(line, "Huge")) fputs(line, stdout);
        if (f) fclose(f);
        f = fopen("/sys/kernel/mm/transparent_hugepage/enabled", "r");
        if (f && fgets(line, sizeof(line), f)) printf("THP: %s", line);
        if (f) fclose(f);
        // the HUGETLB case runs only when the host already has 2 MB pages reserved: the probe changes no host setting
    }
    for (int g = 0; g < G; ++g) { auto c = local_cpus(g); printf("gpu %d local cpus: %zu (first %d)\n", g, c.size(), c.empty() ? -1 : c[0]); }
    std::vector<int> all, lo, hi, one{0};
    for (int g = 0; g < G; ++g) { all.push_back(g); (g < G / 2 ? lo : hi).push_back(g); }
    for (int kind = 0; kind < (getenv("PROBE_ALL_KINDS") ? 4 : 1); ++kind) {
        std::vector<Dev> devs(G);
        bool ok = true;
        for (int g = 0; g < G && ok; ++g) {
            Dev& d = devs[g]; d.id = g;
            CK(cudaSetDevice(g));
            // allocate (first-touch) from a thread bound to the GPU's local CPUs
            std::thread t([&] {
                auto cpus = local_cpus(g);
                if (!cpus.empty()) { cpu_set_t set; CPU_ZERO(&set); for (int c : cpus) CPU_SET(c, &set); pthread_setaffinity_np(pthread_self(), sizeof(set), &set); }
                cudaSetDevice(g);
                d.h_in = host_buf((BufKind)kind, total); d.h_out = host_buf((BufKind)kind, total);
            });
            t.join();
            if (!d.h_in || !d.h_out) { ok = false; break; }
            CK(cudaMalloc(&d.d_in, total)); CK(cudaMalloc(&d.d_out, total));
            CK(cudaStreamCreateWithFlags(&d.s_in, cudaStreamNonBlocking)); CK(cudaStreamCreateWithFlags(&d.s_out, cudaStreamNonBlocking));
        }
        if (!ok) { printf("== %s: unavailable\n", kind_name[kind]); continue; }
        printf("== host buffers: %s\n", kind_name[kind]);
        struct Case { const char* name; const std::vector<int>* act; int mode; size_t chunk; };
        std::vector<Case> cases = {
            {"D2H one GPU, 32 MB", &one, 2, (size_t)32 << 20}, {"H2D one GPU, 32 MB", &one, 1, (size_t)32 << 20},
            {"D2H low half, 32 MB", &lo, 2, (size_t)32 << 20}, {"D2H high half, 32 MB", &hi, 2, (size_t)32 << 20},
            {"D2H all, 32 MB", &all, 2, (size_t)32 << 20}, {"D2H all, 4 MB", &all, 2, (size_t)4 << 20}, {"D2H all, 256 MB", &all, 2, (size_t)256 << 20},
            {"H2D all, 32 MB", &all, 1, (size_t)32 << 20},
            {"both all, 32 MB", &all, 3, (size_t)32 << 20}, {"alternating all, 32 MB", &all, 4, (size_t)32 << 20},
            {"alternating all, 8 MB", &all, 4, (size_t)8 << 20},
        };
        if (kind > 0) cases = {cases[0], cases[4], cases[7], cases[8], cases[9]};
        for (auto& c : cases) {
            if (c.act->empty()) continue;
            auto r = run_case(devs, *c.act, c.mode, c.chunk, total, secs);
            double sum = 0; printf("  %-26s GB/s per direction:", c.name);
            for (int g : *c.act) { printf(" %.1f", r[g]); sum += r[g]; }
            printf(" | sum %.1f\n", sum);
            fflush(stdout);
        }
        if (kind == 0 && G >= 2) {
            // forward results over NVLink to the high half and copy out from there: the high half carries 2x the D2H bytes
            for (int g = 0; g < G; ++g) { CK(cudaSetDevice(g)); for (int p = 0; p < G; ++p) if (p != g) { cudaDeviceEnablePeerAccess(p, 0); cudaGetLastError(); } }
            std::vector<double> rate(G, 0.0); std::vector<std::thread> th; std::atomic<bool> go{false};
            for (int g : hi) th.emplace_back([&, g] {
                Dev& d = devs[g]; Dev& src = devs[g - G / 2];
                CK(cudaSetDevice(d.id)); while (!go.load()) {}
                const size_t chunk = (size_t)32 << 20; const double t0 = now(); size_t moved = 0;
                while (now() - t0 < secs) {
                    for (int rep = 0; rep < 4; ++rep) {
                        CK(cudaMemcpyPeerAsync(d.d_in, d.id, src.d_out, src.id, chunk, d.s_in));        // peer -> me over NVLink
                        CK(cudaMemcpyAsync(d.h_in, d.d_in, chunk, cudaMemcpyDeviceToHost, d.s_in));     // forwarded results out
                        CK(cudaMemcpyAsync(d.h_out, d.d_out, chunk, cudaMemcpyDeviceToHost, d.s_out));  // my own results out
                        moved += 2 * chunk;
                    }
                    CK(cudaStreamSynchronize(d.s_in)); CK(cudaStreamSynchronize(d.s_out));
                }
                rate[g] = moved / (now() - t0) / 1e9;
            });
            go = true; for (auto& t : th) t.join();
            double sum = 0; printf("  %-26s GB/s:", "D2H of all via high half"); for (int g : hi) { printf(" %.1f", rate[g]); sum += rate[g]; } printf(" | sum %.1f\n", sum);
        }
        if (kind == 0 && G >= 8) {
            const std::vector<std::vector<int>> subsets = {{4}, {0, 1}, {4, 5}, {0, 4}, {0, 4, 5, 6, 7}, {0, 1, 4, 5, 6, 7}, {2, 3, 4, 5, 6, 7}};
            for (auto& sub : subsets) {
                auto r = run_case(devs, sub, 2, (size_t)32 << 20, total, secs);
                printf("  D2H subset {"); for (int g : sub) printf("%d ", g); printf("} GB/s:"); double sum = 0;
                for (int g : sub) { printf(" %.1f", r[g]); sum += r[g]; } printf(" | sum %.1f\n", sum); fflush(stdout);
            }
        }
        if (kind == 0 && G >= 2) {
            struct Combo { const char* name; int lo_mode, hi_mode; };
            const Combo combos[] = {{"H2D low only", 1, 0}, {"H2D high only", 0, 1}, {"H2D low + D2H high", 1, 2}, {"H2D high + D2H high", 0, 3},
                                    {"H2D all + D2H high", 1, 3}, {"alternating high only", 0, 4}, {"D2H low + H2D high", 2, 1}};
            for (auto& c : combos) {
                std::vector<int> modes(G), act;
                for (int g = 0; g < G; ++g) { modes[g] = g < G / 2 ? c.lo_mode : c.hi_mode; if (modes[g]) act.push_back(g); }
                auto r = run_case(devs, act, 0, (size_t)32 << 20, total, secs, &modes);
                printf("  %-26s GB/s per direction per active GPU:", c.name);
                for (int g : act) printf(" %.1f(%s)", r[g], modes[g] == 1 ? "in" : modes[g] == 2 ? "out" : "both");
                printf("\n"); fflush(stdout);
            }
        }
        for (auto& d : devs) {
            CK(cudaSetDevice(d.id)); cudaFree(d.d_in); cudaFree(d.d_out);
            if (kind <= 1) { cudaFreeHost(d.h_in); cudaFreeHost(d.h_out); } else { cudaHostUnregister(d.h_in); cudaHostUnregister(d.h_out); munmap(d.h_in, total); munmap(d.h_out, total); }
        }
    }
    return 0;
}
