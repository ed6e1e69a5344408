// cuda_owned.h -- one move-only owner for each kind of CUDA resource the host side holds: device
// buffers, pinned host buffers, events and streams.  An owner records the device that was current when
// it acquired and releases on that device (restoring the thread's device afterwards), so a handle
// that spans several GPUs, or an error return halfway through a set-up, frees everything by going
// out of scope.  Release codes are ignored and nothing here touches the library's error message: the
// call that failed keeps its say.  Owners are host objects only: kernels, views and argument structs
// take the raw pointer from get().  No owner may have static or thread-local storage duration (its
// destructor would run after the CUDA runtime has been torn down at exit).
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>

namespace hs {

// What differs between the kinds: the handle, the call that releases it and, for buffers, the one that acquires.
struct DeviceMem {
    using H = void *;
    static cudaError_t acquire(void **p, size_t bytes, unsigned) { return cudaMalloc(p, bytes); }
    static void release(H p) { cudaFree(p); }
};
struct PinnedMem {
    using H = void *;
    static cudaError_t acquire(void **p, size_t bytes, unsigned flags) { return cudaHostAlloc(p, bytes, flags); }
    static void release(H p) { cudaFreeHost(p); }
};
struct EventRes { using H = cudaEvent_t; static void release(H e) { cudaEventDestroy(e); } };
struct StreamRes { using H = cudaStream_t; static void release(H s) { cudaStreamDestroy(s); } };

template <class K>
class Owned {
  public:
    using H = typename K::H;
    Owned() = default;
    Owned(const Owned &) = delete;
    Owned &operator=(const Owned &) = delete;
    Owned(Owned &&o) noexcept { take(o); }
    Owned &operator=(Owned &&o) noexcept
    {
        if (this != &o) { reset(); take(o); }
        return *this;
    }
    ~Owned() { reset(); }
    H get() const { return h_; }
    void reset()   // release now, on the recorded device; a borrowed handle is only dropped
    {
        if (h_ && !borrowed_) {
            int cur = -1;
            const bool other = cudaGetDevice(&cur) == cudaSuccess && cur != dev_;
            if (other) cudaSetDevice(dev_);
            K::release(h_);
            if (other) cudaSetDevice(cur);
        }
        h_ = H{}; n_ = 0; borrowed_ = false;
    }

  protected:
    cudaError_t adopt(cudaError_t e, H h, size_t n = 0)   // what an acquire returned; on failure stay empty
    {
        if (e == cudaSuccess) { h_ = h; n_ = n; cudaGetDevice(&dev_); }
        return e;
    }
    void take(Owned &o)
    {
        h_ = o.h_; n_ = o.n_; dev_ = o.dev_; borrowed_ = o.borrowed_;
        o.h_ = H{}; o.n_ = 0; o.borrowed_ = false;
    }
    H h_{};
    size_t n_ = 0;            // buffers: capacity in elements
    int dev_ = 0;
    bool borrowed_ = false;   // streams: the caller's, never destroyed here
};

// A buffer of T.  grow(n) keeps the buffer when n elements fit; otherwise it releases it and then
// allocates exactly n (never both at once: peak memory stays at the larger of the two).  A failed
// allocation leaves the owner empty with capacity 0, so nothing dangles and the next call tries again.
template <class T, class K>
class Buffer : public Owned<K> {
  public:
    T *get() const { return static_cast<T *>(this->h_); }
    size_t cap() const { return this->n_; }
    cudaError_t grow(size_t n, unsigned flags = cudaHostAllocDefault)   // flags: pinned buffers only
    {
        if (n <= this->n_) return cudaSuccess;
        this->reset();
        void *p = nullptr;
        const cudaError_t e = K::acquire(&p, n * sizeof(T), flags);   // (before adopt reads p)
        return this->adopt(e, p, n);
    }
};
template <class T> using DevBuf = Buffer<T, DeviceMem>;
template <class T> using PinnedBuf = Buffer<T, PinnedMem>;

struct Event : Owned<EventRes> {
    cudaError_t create(unsigned flags = cudaEventDefault)
    {
        reset();
        cudaEvent_t e = nullptr;
        const cudaError_t r = cudaEventCreateWithFlags(&e, flags);
        return adopt(r, e);
    }
};

struct Stream : Owned<StreamRes> {
    cudaError_t create()   // non-blocking: not ordered against the legacy default stream
    {
        reset();
        cudaStream_t s = nullptr;
        const cudaError_t r = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
        return adopt(r, s);
    }
    void borrow(cudaStream_t s)   // the caller's stream: used, never destroyed
    {
        reset();
        h_ = s;
        borrowed_ = true;
    }
};

}  // namespace hs
