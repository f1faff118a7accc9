// common.cuh -- shared host/device helpers for librcn_cuda (sm_100a only).
#pragma once

#include <cuda_runtime.h>

#include <atomic>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>

#include "../../include/rcn_cuda.h"

namespace rcn {

// ---- error plumbing -----------------------------------------------------------------------------
std::string& last_error_ref();
int fail(int code, const char* fmt, ...);

#define RCN_CUDA_TRY(expr)                                                                        \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess)                                                                    \
            return ::rcn::fail(RCN_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                               __FILE__, __LINE__);                                               \
    } while (0)

#define RCN_TRY(expr)             \
    do {                          \
        int _rc = (expr);         \
        if (_rc != RCN_OK) return _rc; \
    } while (0)

#define RCN_LAUNCH_CHECK()                                                                         \
    do {                                                                                           \
        cudaError_t _e = cudaGetLastError(); /* read and clear: a failed launch is reported once */ \
        if (_e != cudaSuccess)                                                                     \
            return ::rcn::fail(RCN_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), \
                               __FILE__, __LINE__);                                                \
    } while (0)

// ---- launch accounting / built-in per-kernel timing ---------------------------------------------------
// Every kernel launch goes through RCN_LAUNCH: it bumps the process-wide launch counter (bench.py's
// gpu_launches) and, when profiling is enabled (rcn_cuda_profile_enable), brackets the launch with CUDA
// events on the launching stream so bench.py can report per-kernel durations for the roofline.
struct LaunchScope {
    cudaStream_t stream;
    int slot;
    LaunchScope(const char* name, cudaStream_t s);
    ~LaunchScope();
};
#define RCN_LAUNCH(name, stream, ...)                 \
    do {                                              \
        {                                             \
            ::rcn::LaunchScope _ls(name, stream);     \
            __VA_ARGS__;                              \
        }                                             \
        RCN_LAUNCH_CHECK();                           \
    } while (0)

// Is `p` device-accessible memory (device or managed)?  Unregistered host memory reports
// cudaMemoryTypeUnregistered; pinned host memory cudaMemoryTypeHost.
inline bool is_device_ptr(const void* p) {
    if (!p) return false;
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// Grow-only device buffer: steady-state training does no allocation (CUDA-graph friendly).
// Bumped whenever a grow-only device buffer is (re)allocated or released: anything that has baked device pointers into a
// CUDA graph (the host-streaming step graphs, a caller's captured step) compares generations before replaying it.
inline std::atomic<unsigned long long>& alloc_generation() {
    static std::atomic<unsigned long long> g{1};
    return g;
}

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return RCN_OK;
        alloc_generation().fetch_add(1, std::memory_order_relaxed);
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { p = nullptr; return fail(RCN_ERR_CUDA, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e)); }
        cap = want;
        return RCN_OK;
    }
    void release() { if (p) { cudaFree(p); alloc_generation().fetch_add(1, std::memory_order_relaxed); } p = nullptr; cap = 0; }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// Stages a possibly-host input into device memory on `stream`.
struct StagedIn {
    const void* dev = nullptr;
    int stage(const void* src, size_t bytes, DevBuf& scratch, cudaStream_t stream, bool* was_host) {
        if (is_device_ptr(src)) { dev = src; return RCN_OK; }
        RCN_TRY(scratch.reserve(bytes));
        RCN_CUDA_TRY(cudaMemcpyAsync(scratch.p, src, bytes, cudaMemcpyHostToDevice, stream));
        dev = scratch.p;
        if (was_host) *was_host = true;
        return RCN_OK;
    }
};

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per DEVICE: remembers, per kernel call site and device, the
// largest size already granted (one process may drive several GPUs, e.g. rcn_cuda_dp_connect_local).
struct SmemAttrCache {
    size_t granted[64] = {};
    bool need(size_t smem) {
        int d = 0;
        if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= 64) { cudaGetLastError(); return true; }
        if (smem <= granted[d]) return false;
        granted[d] = smem;
        return true;
    }
};

// Scratch of the deterministic two-stage reductions (bias gradient, batch statistics): every CTA leaves a partial, the
// last CTA to arrive (ticket counter, self-resetting) adds the partials in index order.
struct ReduceScratch {
    static constexpr size_t kTicketBytes = 4096;   // 1024 u32 tickets, zeroed when the buffer is (re)allocated
    DevBuf buf;
    int ensure(size_t partial_bytes, cudaStream_t s) {
        const size_t want = kTicketBytes + partial_bytes;
        if (want <= buf.cap) return RCN_OK;
        RCN_TRY(buf.reserve(want));
        RCN_CUDA_TRY(cudaMemsetAsync(buf.p, 0, kTicketBytes, s));
        return RCN_OK;
    }
    unsigned* tickets() const { return buf.as<unsigned>(); }
    double* partials() const { return reinterpret_cast<double*>(buf.as<char>() + kTicketBytes); }
};

// W <- W - (eta/B) * sum  (rcn.rs:214,221): the reference multiplies, rounds, then subtracts (Rust never contracts), so
// the update is NOT a fused multiply-add here either -- given the same gradient sums the new weights are bit-identical.
#ifdef __CUDACC__
__device__ __forceinline__ double sgd_apply(double p, double scale, double g) { return __dsub_rn(p, __dmul_rn(scale, g)); }
#endif

constexpr int kNumSMs = 148;  // B200

inline unsigned cdiv(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }
// Largest gridDim.y / gridDim.z: a launch whose y or z extent grows with the batch caps it and loops, or launches slabs.
constexpr unsigned kMaxGridYZ = 65535;

}  // namespace rcn
