// Error-propagation macros of the C-ABI functions and owning device and page-locked host allocations that only ever
// grow (engine.cu, metric.cu).
#pragma once

#include <cuda_runtime.h>

#include <cstddef>

#include "../../include/vitdet_b200.h"
#include "kernels.h"

#define CU_TRY(expr)                                                                               \
    do {                                                                                           \
        cudaError_t e__ = (expr);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return fail(VITDET_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

#define RC_TRY(expr)                   \
    do {                               \
        int rc__ = (expr);             \
        if (rc__ != 0) return rc__;    \
    } while (0)

namespace vitdet {

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    ~DevBuf() { if (p) cudaFree(p); }
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), bytes(o.bytes) { o.p = nullptr; o.bytes = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) {
            if (p) cudaFree(p);
            p = o.p; bytes = o.bytes; o.p = nullptr; o.bytes = 0;
        }
        return *this;
    }
    int ensure(size_t need) {
        if (need <= bytes) return 0;
        if (p) { cudaFree(p); p = nullptr; bytes = 0; }
        need = (need + 255) / 256 * 256;
        cudaError_t e = cudaMalloc(&p, need);
        if (e != cudaSuccess) return fail(VITDET_E_CUDA, "cudaMalloc(%zu) failed: %s", need, cudaGetErrorString(e));
        bytes = need;
        return 0;
    }
    template <typename T> T* as() const { return static_cast<T*>(p); }
};

// The page-locked host counterpart of DevBuf: staging that cudaMemcpyAsync reads or writes without a bounce
struct PinnedBuf {
    void* p = nullptr;
    size_t bytes = 0;
    ~PinnedBuf() { if (p) cudaFreeHost(p); }
    PinnedBuf() = default;
    PinnedBuf(const PinnedBuf&) = delete;
    PinnedBuf& operator=(const PinnedBuf&) = delete;
    PinnedBuf(PinnedBuf&& o) noexcept : p(o.p), bytes(o.bytes) { o.p = nullptr; o.bytes = 0; }
    PinnedBuf& operator=(PinnedBuf&& o) noexcept {
        if (this != &o) {
            if (p) cudaFreeHost(p);
            p = o.p; bytes = o.bytes; o.p = nullptr; o.bytes = 0;
        }
        return *this;
    }
    int ensure(size_t need) {
        if (need <= bytes) return 0;
        if (p) { cudaFreeHost(p); p = nullptr; bytes = 0; }
        cudaError_t e = cudaHostAlloc(&p, need, cudaHostAllocDefault);
        if (e != cudaSuccess) return fail(VITDET_E_CUDA, "cudaHostAlloc(%zu) failed: %s", need, cudaGetErrorString(e));
        bytes = need;
        return 0;
    }
    template <typename T> T* as() const { return static_cast<T*>(p); }
};

}  // namespace vitdet
