// device_block.h -- a grow-only device allocation, shared by the engine's scratch buffers (engine.cu and its .inc files).
#pragma once
#include <cuda_runtime.h>

#include <cstddef>

namespace dsac {

// reserve(need) keeps the block when it already holds `need` bytes; otherwise it frees it and allocates need + headroom,
// so that the pointer and the size always describe the same live allocation.  No destructor: the block also travels
// by value inside kernel parameter structs (BackwardScratch), so its owner calls release().
struct DeviceBlock {
    void* ptr = nullptr;
    size_t bytes = 0;
    cudaError_t reserve(size_t need, size_t headroom = 0) {
        if (need <= bytes) return cudaSuccess;
        release();
        const cudaError_t st = cudaMalloc(&ptr, need + headroom);
        if (st != cudaSuccess) {
            ptr = nullptr;
            return st;
        }
        bytes = need + headroom;
        return cudaSuccess;
    }
    void release() {
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        bytes = 0;
    }
};

}  // namespace dsac
