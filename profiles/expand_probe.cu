// Host expansion rate of packed FASTQ slabs (scssim_b200/csrc/wire.h) with 1..15 threads, alone and while one stream copies a
// device buffer into pinned memory at the full rate of the GPU's host link (as bench.py's d2h_rate does). Every thread expands its
// own synthetic slab (64 MiB of text: PE150-like records, ~0.1 % verbatim) into its own pinned buffer, as the read stage does.
//   nvcc -O2 -std=c++17 -gencode arch=compute_100a,code=sm_100a -Xcompiler -pthread profiles/expand_probe.cu
//        scssim_b200/csrc/expand_host.cpp -o profiles/expand_probe && profiles/expand_probe [out.json]
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <thread>
#include <vector>

#include "../scssim_b200/csrc/expand_host.h"
#include "../scssim_b200/csrc/wire.h"

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e_)); exit(1); } } while (0)

static double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

struct Slab { std::vector<uint8_t> w; size_t text = 0; char* out = nullptr; };

static Slab make_slab(uint64_t seed, size_t text_target) {
    std::mt19937_64 rng(seed);
    Slab S; S.w.reserve(text_target * 55 / 100);
    uint64_t rec = 0;
    while (S.text < text_target) {
        char hdr[64];
        const int hl = snprintf(hdr, sizeof hdr, "@%u#%u/%d\n", (unsigned)(rng() % 3000000), (unsigned)(rng() % 2000 + 1), (int)(rec & 1) + 1);
        const int np = 150 + (int)(rng() % 7) - 3;
        if (rng() % 1000 == 0) {   // verbatim record
            std::string t(hdr);
            for (int k = 0; k < np; k++) t += "ACGTN"[rng() % 5];
            t += "\n+\n";
            for (int k = 0; k < np; k++) t += (char)('!' + rng() % 42);
            t += "\n";
            S.w.push_back(scs::wire::kVerbatim); S.w.push_back(t.size() & 255); S.w.push_back(t.size() >> 8);
            S.w.insert(S.w.end(), t.begin(), t.end()); S.text += t.size();
        } else {
            S.w.push_back((uint8_t)hl); S.w.push_back(np & 255); S.w.push_back(np >> 8);
            S.w.insert(S.w.end(), hdr, hdr + hl);
            for (int k = 0; k < np; k++) S.w.push_back((uint8_t)((rng() & 3) | ((rng() % 40) << 2)));
            S.text += hl + 2 * np + 4;
        }
        rec++;
    }
    return S;
}

int main(int argc, char** argv) {
    const char* path = argc > 1 ? argv[1] : nullptr;
    const int hw = (int)std::thread::hardware_concurrency();
    const std::vector<int> counts = {1, 2, 4, 8, 12, 15};
    const int maxT = *std::max_element(counts.begin(), counts.end());
    const size_t text = 64ull << 20;
    std::vector<Slab> slabs(maxT);
    for (int t = 0; t < maxT; t++) {
        slabs[t] = make_slab(1000 + t, text);
        CK(cudaMallocHost((void**)&slabs[t].out, slabs[t].text + 64));
        memset(slabs[t].out, 0, slabs[t].text);
        if (scs::expand_wire(slabs[t].w.data(), slabs[t].w.size(), slabs[t].out, '!') != (int64_t)slabs[t].text) { fprintf(stderr, "expand size mismatch\n"); return 1; }
    }
    // device -> pinned copy loop (256 MiB per copy) on its own thread
    const size_t nb = 256ull << 20;
    void* dbuf = nullptr; void* hbuf = nullptr; cudaStream_t st; cudaEvent_t e0, e1;
    CK(cudaMalloc(&dbuf, nb)); CK(cudaMallocHost(&hbuf, nb)); CK(cudaMemset(dbuf, 1, nb)); CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    auto copy_rate = [&](int reps) {
        CK(cudaEventRecord(e0, st));
        for (int r = 0; r < reps; r++) CK(cudaMemcpyAsync(hbuf, dbuf, nb, cudaMemcpyDeviceToHost, st));
        CK(cudaEventRecord(e1, st)); CK(cudaEventSynchronize(e1));
        float ms = 0; CK(cudaEventElapsedTime(&ms, e0, e1));
        return reps * (double)nb / (ms / 1e3) / 1e9;
    };
    copy_rate(2);
    const double link_alone = copy_rate(8);

    auto expand_rate = [&](int T, double& copy_during) {
        std::atomic<bool> stop{false};
        double cbytes = 0, ctime = 0;
        std::thread copier;
        if (copy_during >= 0) copier = std::thread([&] {
            CK(cudaSetDevice(0));
            while (!stop.load()) { const double r = copy_rate(1); cbytes += nb; ctime += nb / (r * 1e9); }
        });
        if (copier.joinable()) std::this_thread::sleep_for(std::chrono::milliseconds(100));
        const int reps = 4;
        std::vector<std::thread> th;
        const double t0 = now();
        for (int t = 0; t < T; t++) th.emplace_back([&, t] { for (int r = 0; r < reps; r++) scs::expand_wire(slabs[t].w.data(), slabs[t].w.size(), slabs[t].out, '!'); });
        for (auto& x : th) x.join();
        const double dt = now() - t0;
        stop = true;
        if (copier.joinable()) { copier.join(); copy_during = cbytes / ctime / 1e9; }
        double bytes = 0; for (int t = 0; t < T; t++) bytes += (double)reps * slabs[t].text;
        return bytes / dt / 1e9;
    };
    char name[256] = "?", power[256] = "?";
    cudaDeviceProp prop; if (cudaGetDeviceProperties(&prop, 0) == cudaSuccess) snprintf(name, sizeof name, "%s", prop.name);
    if (FILE* p = popen("nvidia-smi -i 0 --query-gpu=power.limit --format=csv,noheader 2>/dev/null", "r")) {
        if (fgets(power, sizeof power, p)) power[strcspn(power, "\n")] = 0;
        pclose(p);
    }
    std::string js = "{\"card\": \"" + std::string(name) + "\", \"power_limit\": \"" + power + "\", \"host_cpus\": " + std::to_string(hw) +
                     ", \"avx2\": " + (scs::expand_has_avx2() ? "true" : "false") + ", \"slab_text_MiB\": 64, \"link_alone_GBps\": " + std::to_string(link_alone) + ", \"rows\": [";
    for (size_t i = 0; i < counts.size(); i++) {
        const int T = counts[i];
        double none = -1, during = 0;
        double alone = 0, withc = 0;
        for (int rep = 0; rep < 3; rep++) alone = std::max(alone, expand_rate(T, none));
        double best_copy = 0;
        for (int rep = 0; rep < 3; rep++) { double r = expand_rate(T, during); if (r > withc) { withc = r; best_copy = during; } }
        char row[256];
        snprintf(row, sizeof row, "%s{\"threads\": %d, \"text_GBps_alone\": %.2f, \"text_GBps_with_copy\": %.2f, \"copy_GBps_during\": %.2f}", i ? ", " : "", T, alone, withc, best_copy);
        js += row;
        fprintf(stderr, "threads %2d: %.2f GB/s alone, %.2f GB/s while copying (link %.1f GB/s during, %.1f alone)\n", T, alone, withc, best_copy, link_alone);
    }
    js += "]}\n";
    fputs(js.c_str(), stdout);
    if (path) { FILE* f = fopen(path, "w"); if (f) { fputs(js.c_str(), f); fclose(f); } }
    return 0;
}
