// buffer.h — the owner of every growable allocation of the library: device memory or pinned host memory.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <utility>

// One block of `T`, owned: freed by release() or the destructor, on whichever device is current then.  It converts to
// `T*` (null while nothing is allocated), so kernels, copies and pointer arithmetic take it as they take a pointer.
template <class T, bool Pinned>
class Buffer {
   public:
    Buffer() = default;
    Buffer(const Buffer&) = delete;
    Buffer& operator=(const Buffer&) = delete;
    Buffer(Buffer&& o) noexcept : ptr_(std::exchange(o.ptr_, nullptr)), cap_(std::exchange(o.cap_, 0)) {}
    Buffer& operator=(Buffer&& o) noexcept {
        std::swap(ptr_, o.ptr_);
        std::swap(cap_, o.cap_);
        return *this;
    }
    ~Buffer() { release(); }

    // When `need` bytes exceed the capacity: frees the block and allocates `alloc_if_grown` bytes (>= need).  The
    // contents are discarded then; on failure the buffer is empty.
    cudaError_t reserve(size_t need, size_t alloc_if_grown) {
        if (need <= cap_) return cudaSuccess;
        release();
        void* p = nullptr;
        const cudaError_t e = Pinned ? cudaHostAlloc(&p, alloc_if_grown, cudaHostAllocDefault) : cudaMalloc(&p, alloc_if_grown);
        if (e != cudaSuccess) return e;
        ptr_ = static_cast<T*>(p);
        cap_ = alloc_if_grown;
        return cudaSuccess;
    }
    cudaError_t reserve(size_t need) { return reserve(need, need); }

    void release() {
        if (ptr_) Pinned ? cudaFreeHost(ptr_) : cudaFree(ptr_);
        ptr_ = nullptr;
        cap_ = 0;
    }

    T* get() const { return ptr_; }
    operator T*() const { return ptr_; }
    size_t capacity() const { return cap_; }  // bytes

   private:
    T* ptr_ = nullptr;
    size_t cap_ = 0;
};

template <class T>
using DeviceBuffer = Buffer<T, false>;
template <class T>
using PinnedBuffer = Buffer<T, true>;
