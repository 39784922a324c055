// See hostpool.hpp.
#include "hostpool.hpp"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include <sched.h>

namespace aptb200 {

static std::vector<int> parse_cpulist(const std::string &s) {
    std::vector<int> cpus;
    size_t i = 0;
    while (i < s.size()) {
        char *end = nullptr;
        const long a = strtol(s.c_str() + i, &end, 10);
        if (end == s.c_str() + i) break;
        long b = a;
        i = static_cast<size_t>(end - s.c_str());
        if (i < s.size() && s[i] == '-') {
            b = strtol(s.c_str() + i + 1, &end, 10);
            i = static_cast<size_t>(end - s.c_str());
        }
        for (long c = a; c <= b && c < 4096; ++c) cpus.push_back(static_cast<int>(c));
        if (i < s.size() && s[i] == ',') ++i; else break;
    }
    return cpus;
}

std::vector<int> device_local_cpus(int device) {
    char bus[64] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device) != cudaSuccess) {
        cudaGetLastError();
        return {};
    }
    for (char *p = bus; *p; ++p) *p = static_cast<char>(tolower(*p));
    const std::string path = std::string("/sys/bus/pci/devices/") + bus + "/local_cpulist";
    FILE *f = fopen(path.c_str(), "r");
    if (!f) return {};
    char line[4096] = {0};
    const bool got = fgets(line, sizeof(line), f) != nullptr;
    fclose(f);
    if (!got) return {};
    return parse_cpulist(line);
}

bool bind_thread_to_device(int device) {
    if (getenv("APTB200_NO_AFFINITY")) return false;
    const std::vector<int> cpus = device_local_cpus(device);
    if (cpus.empty()) return false;
    cpu_set_t allowed, want;
    CPU_ZERO(&allowed);
    if (sched_getaffinity(0, sizeof(allowed), &allowed) != 0) return false;
    CPU_ZERO(&want);
    int n = 0;
    for (int c : cpus)
        if (c < CPU_SETSIZE && CPU_ISSET(c, &allowed)) { CPU_SET(c, &want); ++n; }   // stay inside the cgroup / taskset mask
    if (n == 0) return false;
    return sched_setaffinity(0, sizeof(want), &want) == 0;
}

// --------------------------------------------------------------------------------------------- CopyPool

CopyPool::CopyPool(int threads, int device) : device_(device) {
    for (int t = 1; t < threads; ++t) workers_.emplace_back([this, t] { worker(t); });
}

CopyPool::~CopyPool() {
    {
        std::lock_guard<std::mutex> lk(m_);
        quit_.store(true, std::memory_order_release);
        gen_atomic_.fetch_add(1, std::memory_order_acq_rel);
    }
    cv_start_.notify_all();
    for (auto &w : workers_) w.join();
}

void CopyPool::worker(int index) {
    bind_thread_to_device(device_);
    uint64_t seen = 0;
    for (;;) {
        // chunks of one upload follow each other within ~0.3 ms: spin that long before going to sleep on the condition
        // variable (a futex wake-up costs 50-100 us, twice per chunk)
        const auto t0 = std::chrono::steady_clock::now();
        while (gen_atomic_.load(std::memory_order_acquire) == seen) {
            if (std::chrono::steady_clock::now() - t0 > std::chrono::microseconds(500)) {
                std::unique_lock<std::mutex> lk(m_);
                cv_start_.wait(lk, [&] { return gen_atomic_.load(std::memory_order_acquire) != seen; });
                break;
            }
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
        }
        seen = gen_atomic_.load(std::memory_order_acquire);
        if (quit_.load(std::memory_order_acquire)) return;
        const size_t a = std::min(bytes_, slice_ * static_cast<size_t>(index));
        const size_t b = std::min(bytes_, a + slice_);
        if (b > a) memcpy(dst_ + a, src_ + a, b - a);
        pending_.fetch_sub(1, std::memory_order_acq_rel);
    }
}

void CopyPool::copy(void *dst, const void *src, size_t bytes) {
    const size_t n = workers_.size() + 1;
    if (bytes < (256u << 10) || n == 1) {
        memcpy(dst, src, bytes);
        return;
    }
    size_t slice;
    {
        std::lock_guard<std::mutex> lk(m_);                   // also orders the job fields before the generation bump
        slice = slice_ = ((bytes + n - 1) / n + 4095) & ~static_cast<size_t>(4095);
        dst_ = static_cast<char *>(dst);
        src_ = static_cast<const char *>(src);
        bytes_ = bytes;
        pending_.store(static_cast<int>(workers_.size()), std::memory_order_release);
        gen_atomic_.fetch_add(1, std::memory_order_acq_rel);
    }
    cv_start_.notify_all();
    memcpy(dst, src, std::min(bytes, slice));                 // the caller's thread takes slice 0
    while (pending_.load(std::memory_order_acquire) != 0) {   // the workers finish within microseconds of this thread
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
    }
}

// --------------------------------------------------------------------------------------------- HostStager

HostStager::HostStager(int device, size_t chunk_bytes, int ring, int threads)
    : device_(device), chunk_(chunk_bytes), pool_(threads, device) {
    ring_.assign(ring, nullptr);
    ev_.assign(ring, nullptr);
    used_.assign(ring, false);
    ok_ = true;
    for (int i = 0; i < ring; ++i) {
        // write-combined pinned staging: the copy threads only ever write it (streaming stores) and only the DMA engine
        // reads it -- 4.3 ms instead of 5.2 ms per 172.8 MB recording through apt_decode (APTB200_COPY_NO_WC=1 reverts)
        static const bool wc = getenv("APTB200_COPY_NO_WC") == nullptr;
        if (cudaHostAlloc(reinterpret_cast<void **>(&ring_[i]), chunk_, wc ? cudaHostAllocWriteCombined : cudaHostAllocDefault) != cudaSuccess ||
            cudaEventCreateWithFlags(&ev_[i], cudaEventDisableTiming) != cudaSuccess) {
            cudaGetLastError();
            ok_ = false;
            break;
        }
        memset(ring_[i], 0, chunk_);                          // touch: the pages land on the node of this thread
    }
}

HostStager::~HostStager() {
    for (auto e : ev_)
        if (e) cudaEventDestroy(e);
    for (auto p : ring_)
        if (p) cudaFreeHost(p);
}

cudaError_t HostStager::upload(void *dst, const void *src, size_t bytes, cudaStream_t stream) {
    static const bool trace = getenv("APTB200_TRACE_HOST") != nullptr;
    const auto t_begin = std::chrono::steady_clock::now();
    double t_wait = 0, t_copy = 0;
    size_t off = 0;
    size_t c = 0;
    const size_t nr = ring_.size();
    while (off < bytes) {
        const size_t nb = std::min(chunk_, bytes - off);
        const size_t r = c % nr;
        const auto t0 = std::chrono::steady_clock::now();
        if (used_[r]) {
            const cudaError_t e = cudaEventSynchronize(ev_[r]);   // the DMA that last read this buffer has finished
            if (e != cudaSuccess) return e;
        }
        const auto t1 = std::chrono::steady_clock::now();
        pool_.copy(ring_[r], static_cast<const char *>(src) + off, nb);
        if (trace) {
            t_wait += std::chrono::duration<double>(t1 - t0).count();
            t_copy += std::chrono::duration<double>(std::chrono::steady_clock::now() - t1).count();
        }
        cudaError_t e = cudaMemcpyAsync(static_cast<char *>(dst) + off, ring_[r], nb, cudaMemcpyHostToDevice, stream);
        if (e != cudaSuccess) return e;
        e = cudaEventRecord(ev_[r], stream);
        if (e != cudaSuccess) return e;
        used_[r] = true;
        off += nb;
        ++c;
    }
    if (trace)
        fprintf(stderr, "[aptb200 host] upload %.1f MB in %zu chunks: %.2f ms (ring waits %.2f ms, memcpy %.2f ms = %.1f GB/s, %d threads)\n",
                bytes / 1e6, c, std::chrono::duration<double>(std::chrono::steady_clock::now() - t_begin).count() * 1e3, t_wait * 1e3,
                t_copy * 1e3, bytes / t_copy / 1e9, pool_.threads());
    return cudaSuccess;
}

bool is_pageable(const void *p) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return at.type == cudaMemoryTypeUnregistered;
}

}  // namespace aptb200
