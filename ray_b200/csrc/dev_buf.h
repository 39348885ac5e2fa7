// dev_buf.h -- DevBuf<T>: the single owner of one device allocation (host code only).
//
// The destructor frees the block; the owner of a DevBuf makes sure its device is current when that happens.  Move-only.
#pragma once

#include <stddef.h>

#include <utility>

#include <cuda_runtime.h>

template <typename T> class DevBuf {
  public:
    DevBuf() = default;
    DevBuf(DevBuf &&o) noexcept : p_(std::exchange(o.p_, nullptr)), n_(std::exchange(o.n_, 0)) {}
    DevBuf &operator=(DevBuf &&o) noexcept {
        if (this != &o) {
            reset();
            p_ = std::exchange(o.p_, nullptr);
            n_ = std::exchange(o.n_, 0);
        }
        return *this;
    }
    ~DevBuf() { reset(); }

    // n elements, contents undefined.  The old block is freed BEFORE the new one is requested, so a resize never holds
    // both; n == 0 or a failure leaves the buffer empty.
    cudaError_t alloc(size_t n) {
        reset();
        if (n == 0) {
            return cudaSuccess;
        }
        const cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&p_), n * sizeof(T));
        if (e != cudaSuccess) {
            p_ = nullptr;
            return e;
        }
        n_ = n;
        return cudaSuccess;
    }

    void reset() {
        if (p_) {
            cudaFree(p_);
        }
        p_ = nullptr;
        n_ = 0;
    }

    T *get() const { return p_; }
    size_t count() const { return n_; }

  private:
    T *p_ = nullptr;
    size_t n_ = 0;
};
