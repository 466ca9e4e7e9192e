// rt_buffer.h — one growable allocation owned by the library: device memory, or page-locked host memory (host code only).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

namespace rt {

enum class Mem { Device, Pinned };

template <typename T, Mem M = Mem::Device>
struct Buffer {
    T *ptr = nullptr;
    size_t cap = 0;           // elements

    Buffer() = default;
    Buffer(const Buffer &) = delete;
    Buffer &operator=(const Buffer &) = delete;
    ~Buffer() { release(); }

    // At least `need` elements.  A smaller buffer is freed and need + slack elements are allocated; the contents are not kept.
    // On failure the buffer is empty and the error is returned, so the next call allocates again.
    cudaError_t reserve(size_t need, size_t slack = 0) {
        if (need <= cap) return cudaSuccess;
        release();
        void *p = nullptr;
        cudaError_t e;
        if constexpr (M == Mem::Device) e = cudaMalloc(&p, (need + slack) * sizeof(T));
        else e = cudaMallocHost(&p, (need + slack) * sizeof(T));
        if (e != cudaSuccess) return e;
        ptr = static_cast<T *>(p);
        cap = need + slack;
        return cudaSuccess;
    }

private:
    void release() {
        if (!ptr) return;
        if constexpr (M == Mem::Device) cudaFree(ptr);
        else cudaFreeHost(ptr);
        ptr = nullptr;
        cap = 0;
    }
};

}  // namespace rt
