// devbuf.hpp — the one owner of every device and pinned-host allocation of tuna_b200.cu.
//
// A Buf holds one cudaMalloc'd (or cudaMallocHost'd) array, frees it in its destructor and is move-only.  Moving keeps the address:
// job descriptors, class-table views and kernel arguments hold raw pointers into buffers that live in vectors and maps.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <string>
#include <utility>

#include "../../include/tuna_b200.h"

namespace tuna {

template <typename T, bool Pinned>
class Buf {
public:
    Buf() = default;
    Buf(const Buf&) = delete;
    Buf& operator=(const Buf&) = delete;
    Buf(Buf&& o) noexcept : p_(std::exchange(o.p_, nullptr)), n_(std::exchange(o.n_, 0)) {}
    Buf& operator=(Buf&& o) noexcept {
        if (this != &o) { reset(); p_ = std::exchange(o.p_, nullptr); n_ = std::exchange(o.n_, 0); }
        return *this;
    }
    ~Buf() { reset(); }

    // At least count elements.  A buffer that is large enough stays where it is; otherwise the old one is freed BEFORE exactly count
    // elements are allocated (the peak stays one copy of the n^4 tensors).  On failure the buffer is empty, err says why, and the
    // result is TUNA_ERR_NOMEM.
    int grow(size_t count, std::string& err) {
        if (count <= n_) return TUNA_OK;
        reset();
        void* q = nullptr;
        const cudaError_t e = Pinned ? cudaMallocHost(&q, count * sizeof(T)) : cudaMalloc(&q, count * sizeof(T));
        if (e != cudaSuccess) {
            cudaGetLastError();
            err = Pinned ? std::string("pinned host allocation failed")
                         : "cudaMalloc of " + std::to_string(count * sizeof(T)) + " bytes failed: " + cudaGetErrorString(e);
            return TUNA_ERR_NOMEM;
        }
        p_ = static_cast<T*>(q);
        n_ = count;
        return TUNA_OK;
    }
    void reset() {
        if (p_) { if (Pinned) cudaFreeHost(p_); else cudaFree(p_); }
        p_ = nullptr;
        n_ = 0;
    }
    T* get() const { return p_; }
    size_t capacity() const { return n_; }
    operator T*() const { return p_; }

private:
    T* p_ = nullptr;
    size_t n_ = 0;
};

template <typename T> using DevBuf = Buf<T, false>;
template <typename T> using PinnedBuf = Buf<T, true>;

}  // namespace tuna
