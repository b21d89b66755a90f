// Host-side plumbing shared by the C-ABI translation units: the error record behind dvbs2fec_last_error, the CUDA
// call check, device and page-locked buffers that free themselves, and the synchronous upload of host tables.
#pragma once
#include <cstddef>
#include <utility>

#include <cuda_runtime.h>

#include "../../include/dvbs2fec.h"

namespace s2 {

// Records the message that dvbs2fec_last_error returns (per thread) and returns code.  Defined in api.cu.
int fail(int code, const char* fmt, ...) __attribute__((format(printf, 2, 3)));

#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return s2::fail(DVBS2FEC_ECUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// cap elements of device (Pinned = false) or page-locked host memory, freed with the buffer.  The owner of a device
// buffer makes its device current before the buffer goes.
template <typename T, bool Pinned>
struct CudaBuf {
    T* p = nullptr;
    size_t cap = 0;
    CudaBuf() = default;
    CudaBuf(CudaBuf&& o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
    CudaBuf& operator=(CudaBuf&& o) noexcept {
        std::swap(p, o.p);
        std::swap(cap, o.cap);
        return *this;
    }
    ~CudaBuf() { drop(); }
    // at least n elements; the contents are discarded when it grows
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        drop();
        cudaError_t e = Pinned ? cudaMallocHost(&p, n * sizeof(T)) : cudaMalloc(&p, n * sizeof(T));
        if (e == cudaSuccess) cap = n;
        else p = nullptr;
        return e;
    }
    // device buffers: at least n elements, the first `keep` kept (copied on st, which is then synchronised)
    cudaError_t grow(size_t n, size_t keep, cudaStream_t st) {
        if (n <= cap) return cudaSuccess;
        T* q = nullptr;
        cudaError_t e = cudaMalloc(&q, n * sizeof(T));
        if (e != cudaSuccess) return e;
        if (p && keep) e = cudaMemcpyAsync(q, p, keep * sizeof(T), cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        drop();
        p = q;
        cap = n;
        return e;
    }

private:
    void drop() {
        if (p) {
            if (Pinned) cudaFreeHost(p);
            else cudaFree(p);
        }
        p = nullptr;
        cap = 0;
    }
};
template <typename T>
using DevBuf = CudaBuf<T, false>;
template <typename T>
using PinBuf = CudaBuf<T, true>;

// Host data into device memory, synchronously: a cudaMemcpy from pageable memory returns once the data are staged,
// and the library's non-blocking streams do not wait for the default stream.
inline cudaError_t upload(void* dst, const void* src, size_t bytes) {
    cudaError_t e = cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice);
    return e == cudaSuccess ? cudaStreamSynchronize(nullptr) : e;
}

}  // namespace s2
