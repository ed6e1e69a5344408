// tests/host_emul/cuda_count.cpp -- TEST INFRASTRUCTURE (LD_PRELOAD interposer, tests/test_gpu_lifecycle.py).
// Counts live device buffers, pinned buffers, events and streams acquired through the CUDA runtime's
// public calls, and forwards every call unchanged to the real runtime (dlsym(RTLD_NEXT)): results are
// never altered.  libhymet_screen.so links cudart shared, so its calls resolve here first.
#include <cuda_runtime_api.h>
#include <dlfcn.h>
#include <stdint.h>

#include <mutex>
#include <set>

namespace {
std::mutex g_mu;
std::set<uintptr_t> g_live[4];   // device buffers, pinned buffers, events, streams

// the runtime's own entry point: next in the global scope, or in the already loaded libcudart when the
// library that needs it was dlopen()ed locally (ctypes)
template <class F> F real(const char *name)
{
    void *f = dlsym(RTLD_NEXT, name);
    if (!f) {
        void *h = dlopen("libcudart.so.12", RTLD_NOW | RTLD_NOLOAD);
        if (h) f = dlsym(h, name);
    }
    return reinterpret_cast<F>(f);
}
void add(int k, const void *h)
{
    std::lock_guard<std::mutex> lk(g_mu);
    g_live[k].insert((uintptr_t)h);
}
void drop(int k, const void *h)
{
    std::lock_guard<std::mutex> lk(g_mu);
    g_live[k].erase((uintptr_t)h);
}
}  // namespace

extern "C" {

int cuda_count_live(int kind)
{
    std::lock_guard<std::mutex> lk(g_mu);
    return (int)g_live[kind].size();
}

cudaError_t cudaMalloc(void **p, size_t n)
{
    static auto f = real<cudaError_t (*)(void **, size_t)>("cudaMalloc");
    const cudaError_t e = f(p, n);
    if (e == cudaSuccess && *p) add(0, *p);
    return e;
}
cudaError_t cudaFree(void *p)
{
    static auto f = real<cudaError_t (*)(void *)>("cudaFree");
    const cudaError_t e = f(p);
    if (e == cudaSuccess && p) drop(0, p);
    return e;
}
cudaError_t cudaHostAlloc(void **p, size_t n, unsigned int flags)
{
    static auto f = real<cudaError_t (*)(void **, size_t, unsigned int)>("cudaHostAlloc");
    const cudaError_t e = f(p, n, flags);
    if (e == cudaSuccess && *p) add(1, *p);
    return e;
}
cudaError_t cudaMallocHost(void **p, size_t n)
{
    static auto f = real<cudaError_t (*)(void **, size_t)>("cudaMallocHost");
    const cudaError_t e = f(p, n);
    if (e == cudaSuccess && *p) add(1, *p);
    return e;
}
cudaError_t cudaFreeHost(void *p)
{
    static auto f = real<cudaError_t (*)(void *)>("cudaFreeHost");
    const cudaError_t e = f(p);
    if (e == cudaSuccess && p) drop(1, p);
    return e;
}
cudaError_t cudaEventCreate(cudaEvent_t *ev)
{
    static auto f = real<cudaError_t (*)(cudaEvent_t *)>("cudaEventCreate");
    const cudaError_t e = f(ev);
    if (e == cudaSuccess) add(2, *ev);
    return e;
}
cudaError_t cudaEventCreateWithFlags(cudaEvent_t *ev, unsigned int flags)
{
    static auto f = real<cudaError_t (*)(cudaEvent_t *, unsigned int)>("cudaEventCreateWithFlags");
    const cudaError_t e = f(ev, flags);
    if (e == cudaSuccess) add(2, *ev);
    return e;
}
cudaError_t cudaEventDestroy(cudaEvent_t ev)
{
    static auto f = real<cudaError_t (*)(cudaEvent_t)>("cudaEventDestroy");
    const cudaError_t e = f(ev);
    if (e == cudaSuccess) drop(2, ev);
    return e;
}
cudaError_t cudaStreamCreate(cudaStream_t *st)
{
    static auto f = real<cudaError_t (*)(cudaStream_t *)>("cudaStreamCreate");
    const cudaError_t e = f(st);
    if (e == cudaSuccess) add(3, *st);
    return e;
}
cudaError_t cudaStreamCreateWithFlags(cudaStream_t *st, unsigned int flags)
{
    static auto f = real<cudaError_t (*)(cudaStream_t *, unsigned int)>("cudaStreamCreateWithFlags");
    const cudaError_t e = f(st, flags);
    if (e == cudaSuccess) add(3, *st);
    return e;
}
cudaError_t cudaStreamDestroy(cudaStream_t st)
{
    static auto f = real<cudaError_t (*)(cudaStream_t)>("cudaStreamDestroy");
    const cudaError_t e = f(st);
    if (e == cudaSuccess) drop(3, st);
    return e;
}

}  // extern "C"
