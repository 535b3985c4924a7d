// cuda_owned.hpp — owning handles for the chain engine's CUDA resources (host code only).
//
// DeviceArray / PinnedArray own a cudaMalloc / cudaMallocHost array; size() is its capacity in elements.  There is never a
// capacity without memory behind it: a failed alloc() or grow() leaves the array empty (null, size 0), so a call that
// reported the error can be retried, and nothing is freed twice.  Event and Stream destroy their handle.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>
#include <memory>
#include <type_traits>
#include <utility>

namespace iqgpu {

template <typename T, bool Pinned>
class CudaArray {
public:
    CudaArray() = default;
    CudaArray(CudaArray&& o) noexcept : p_(std::exchange(o.p_, nullptr)), n_(std::exchange(o.n_, 0)) {}
    CudaArray& operator=(CudaArray&& o) noexcept
    {
        if (this != &o) { reset(); p_ = std::exchange(o.p_, nullptr); n_ = std::exchange(o.n_, 0); }
        return *this;
    }
    ~CudaArray() { reset(); }

    T* data() const { return p_; }
    size_t size() const { return n_; }
    void reset()
    {
        if (p_) { if (Pinned) cudaFreeHost(p_); else cudaFree(p_); }
        p_ = nullptr; n_ = 0;
    }
    // frees what the array held, then allocates n elements
    cudaError_t alloc(size_t n)
    {
        reset();
        void* p = nullptr;
        cudaError_t e = n > SIZE_MAX / sizeof(T) ? cudaErrorMemoryAllocation
                                                 : (Pinned ? cudaMallocHost(&p, n * sizeof(T)) : cudaMalloc(&p, n * sizeof(T)));
        if (e != cudaSuccess) {
            cudaGetLastError();     // reported here: a later launch check must not see it again
            return e;
        }
        p_ = static_cast<T*>(p); n_ = n;
        return cudaSuccess;
    }
    // nothing when `need` elements fit; else drain() (whatever may still use the array has finished), free, allocate `cap`
    template <typename Drain>
    cudaError_t grow(size_t need, size_t cap, Drain&& drain)
    {
        if (need <= n_) return cudaSuccess;
        const cudaError_t e = drain();
        if (e != cudaSuccess) { reset(); return e; }
        return alloc(cap);
    }

private:
    T* p_ = nullptr;
    size_t n_ = 0;
};
template <typename T> using DeviceArray = CudaArray<T, false>;
template <typename T> using PinnedArray = CudaArray<T, true>;

// drain of a grow() whose old memory nothing can still be using
inline cudaError_t no_drain() { return cudaSuccess; }

// owning runtime handle; converts to the raw handle, so it passes straight to the runtime API
template <typename H, cudaError_t (*Destroy)(H)>
struct Destroyer { void operator()(H h) const { Destroy(h); } };
template <typename H, cudaError_t (*Destroy)(H)>
struct Owned : std::unique_ptr<std::remove_pointer_t<H>, Destroyer<H, Destroy>> {
    operator H() const { return this->get(); }
};
using Event = Owned<cudaEvent_t, cudaEventDestroy>;
using Stream = Owned<cudaStream_t, cudaStreamDestroy>;

inline cudaError_t create(Event& ev, unsigned flags = cudaEventDisableTiming)
{
    cudaEvent_t h = nullptr;
    const cudaError_t e = cudaEventCreateWithFlags(&h, flags);
    if (e == cudaSuccess) ev.reset(h);
    return e;
}
inline cudaError_t create(Stream& s)
{
    cudaStream_t h = nullptr;
    const cudaError_t e = cudaStreamCreateWithFlags(&h, cudaStreamNonBlocking);
    if (e == cudaSuccess) s.reset(h);
    return e;
}

}  // namespace iqgpu
