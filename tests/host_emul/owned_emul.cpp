// tests/host_emul/owned_emul.cpp -- TEST INFRASTRUCTURE.
// Compiles csrc/cuda_owned.h with g++ against a fake CUDA runtime defined here: the fake hands out
// made-up handles, tracks which are live per kind and the thread's current device, records the device
// every release happens on, and can fail the n-th acquisition.  Nothing touches a GPU.  Each check_*
// returns 0, or the line of the first expectation that did not hold.
#include <stdint.h>

#include <map>
#include <type_traits>
#include <utility>
#include <vector>

#include "../../hymet_b200/csrc/cuda_owned.h"

using namespace hs;

namespace {

enum Kind { kDev, kPinned, kEvent, kStream, kKinds };
std::map<uintptr_t, Kind> g_live;        // handle -> kind
std::vector<int> g_release_dev;          // device current at each release
int g_device = 0, g_acquired = 0, g_fail_at = -1;   // fail_at: index of the acquisition that fails
uintptr_t g_next = 0x1000;

cudaError_t acquire(Kind k, uintptr_t *h)
{
    if (g_acquired++ == g_fail_at) return cudaErrorMemoryAllocation;
    *h = (g_next += 0x100);
    g_live[*h] = k;
    return cudaSuccess;
}
cudaError_t release(Kind k, uintptr_t h)
{
    auto it = g_live.find(h);
    if (!h || it == g_live.end() || it->second != k) return cudaErrorInvalidValue;   // double or foreign release
    g_live.erase(it);
    g_release_dev.push_back(g_device);
    return cudaSuccess;
}
int live(Kind k)
{
    int n = 0;
    for (auto &e : g_live) n += e.second == k;
    return n;
}
void restart()
{
    g_live.clear(); g_release_dev.clear();
    g_device = 0; g_acquired = 0; g_fail_at = -1;
}

}  // namespace

extern "C" {
cudaError_t cudaMalloc(void **p, size_t) { uintptr_t h = 0; cudaError_t e = acquire(kDev, &h); *p = (void *)h; return e; }
cudaError_t cudaFree(void *p) { return p ? release(kDev, (uintptr_t)p) : cudaSuccess; }
cudaError_t cudaHostAlloc(void **p, size_t, unsigned int) { uintptr_t h = 0; cudaError_t e = acquire(kPinned, &h); *p = (void *)h; return e; }
cudaError_t cudaFreeHost(void *p) { return release(kPinned, (uintptr_t)p); }
cudaError_t cudaEventCreateWithFlags(cudaEvent_t *ev, unsigned int)
{
    uintptr_t h = 0; cudaError_t e = acquire(kEvent, &h); *ev = (cudaEvent_t)h; return e;
}
cudaError_t cudaEventDestroy(cudaEvent_t ev) { return release(kEvent, (uintptr_t)ev); }
cudaError_t cudaStreamCreateWithFlags(cudaStream_t *st, unsigned int)
{
    uintptr_t h = 0; cudaError_t e = acquire(kStream, &h); *st = (cudaStream_t)h; return e;
}
cudaError_t cudaStreamDestroy(cudaStream_t st) { return release(kStream, (uintptr_t)st); }
cudaError_t cudaGetDevice(int *d) { *d = g_device; return cudaSuccess; }
cudaError_t cudaSetDevice(int d) { g_device = d; return cudaSuccess; }
}

static_assert(!std::is_copy_constructible<DevBuf<int>>::value && !std::is_copy_assignable<DevBuf<int>>::value, "owners do not copy");
static_assert(!std::is_copy_constructible<PinnedBuf<int>>::value && !std::is_copy_assignable<PinnedBuf<int>>::value, "owners do not copy");
static_assert(!std::is_copy_constructible<Event>::value && !std::is_copy_assignable<Event>::value, "owners do not copy");
static_assert(!std::is_copy_constructible<Stream>::value && !std::is_copy_assignable<Stream>::value, "owners do not copy");
static_assert(std::is_nothrow_move_constructible<DevBuf<int>>::value && std::is_nothrow_move_assignable<DevBuf<int>>::value &&
                  std::is_nothrow_move_constructible<Event>::value && std::is_nothrow_move_constructible<Stream>::value,
              "moves are noexcept: std::vector growth moves instead of copying");

#define EXPECT(c) do { if (!(c)) return __LINE__; } while (0)

extern "C" {

// move-construct, move-assign, self-move and std::vector growth release each resource exactly once
int check_moves()
{
    restart();
    {
        DevBuf<int> a;
        EXPECT(a.grow(10) == cudaSuccess && a.get() && a.cap() == 10 && live(kDev) == 1);
        DevBuf<int> b(std::move(a));
        EXPECT(!a.get() && a.cap() == 0 && b.cap() == 10 && live(kDev) == 1);
        DevBuf<int> c;
        EXPECT(c.grow(5) == cudaSuccess && live(kDev) == 2);
        c = std::move(b);   // c's own buffer goes, b's moves in
        EXPECT(live(kDev) == 1 && g_release_dev.size() == 1 && c.cap() == 10 && !b.get());
        DevBuf<int> &alias = c;
        c = std::move(alias);
        EXPECT(live(kDev) == 1 && c.get() && c.cap() == 10);
        Event e;
        EXPECT(e.create() == cudaSuccess);
        Event f = std::move(e);
        EXPECT(live(kEvent) == 1 && !e.get() && f.get());
        std::vector<PinnedBuf<char>> v;
        for (int i = 0; i < 100; i++) {
            PinnedBuf<char> p;
            EXPECT(p.grow(64) == cudaSuccess);
            v.push_back(std::move(p));
        }
        std::vector<Event> evs(3);
        for (auto &x : evs) EXPECT(x.create() == cudaSuccess);
        evs.reserve(1000);
        EXPECT(live(kPinned) == 100 && live(kEvent) == 4 && g_release_dev.size() == 1);
    }
    EXPECT(g_live.empty());
    EXPECT(g_release_dev.size() == 1 + 1 + 1 + 100 + 3);   // c's first, c's second, the event, 100 pinned, 3 events
    return 0;
}

// grow keeps a buffer that fits; a failed grow leaves the owner empty with capacity 0 and nothing
// live, and the next grow succeeds
int check_grow()
{
    restart();
    DevBuf<double> a;
    EXPECT(a.grow(0) == cudaSuccess && !a.get() && g_acquired == 0);
    EXPECT(a.grow(100) == cudaSuccess && a.cap() == 100);
    void *first = a.get();
    EXPECT(a.grow(100) == cudaSuccess && a.grow(7) == cudaSuccess && a.get() == first && g_acquired == 1);
    g_fail_at = g_acquired;
    EXPECT(a.grow(101) == cudaErrorMemoryAllocation);
    EXPECT(!a.get() && a.cap() == 0 && live(kDev) == 0);
    EXPECT(a.grow(50) == cudaSuccess && a.get() && a.cap() == 50 && live(kDev) == 1);
    PinnedBuf<char> p;
    g_fail_at = g_acquired;
    EXPECT(p.grow(8, cudaHostAllocMapped) == cudaErrorMemoryAllocation && !p.get() && p.cap() == 0 && live(kPinned) == 0);
    EXPECT(p.grow(8, cudaHostAllocMapped) == cudaSuccess && live(kPinned) == 1);
    Event e;
    g_fail_at = g_acquired;
    EXPECT(e.create() == cudaErrorMemoryAllocation && !e.get() && live(kEvent) == 0);
    EXPECT(e.create() == cudaSuccess && e.get() && live(kEvent) == 1);
    a.reset(); p.reset(); e.reset();
    EXPECT(g_live.empty());
    return 0;
}

// release on the device that was current at acquisition, then the caller's device again
int check_devices()
{
    restart();
    {
        g_device = 3;
        DevBuf<int> a;
        EXPECT(a.grow(4) == cudaSuccess);
        g_device = 5;
        Event e;
        EXPECT(e.create() == cudaSuccess);
        Stream s;
        EXPECT(s.create() == cudaSuccess);
        g_device = 1;
        a.reset();
        EXPECT(g_release_dev.back() == 3 && g_device == 1);
        g_device = 3;
        DevBuf<int> b;
        EXPECT(b.grow(4) == cudaSuccess);
        g_device = 0;
        DevBuf<int> c(std::move(b));   // the device travels with the buffer
        g_device = 7;
    }
    EXPECT(g_device == 7 && g_live.empty());
    // reverse order of declaration: c (device 3), s and e (device 5)
    EXPECT(g_release_dev.size() == 4 && g_release_dev[1] == 3 && g_release_dev[2] == 5 && g_release_dev[3] == 5);
    return 0;
}

// a borrowed stream is never destroyed: not on reset, re-borrow, create, move or destruction
int check_borrowed_stream()
{
    restart();
    cudaStream_t theirs = nullptr;
    EXPECT(cudaStreamCreateWithFlags(&theirs, 0) == cudaSuccess);
    {
        Stream s;
        EXPECT(s.create() == cudaSuccess && live(kStream) == 2);
        s.borrow(theirs);   // the handle's own stream goes, the caller's is used
        EXPECT(s.get() == theirs && live(kStream) == 1);
        Stream t(std::move(s));
        EXPECT(t.get() == theirs && !s.get());
        t.reset();
        EXPECT(!t.get() && live(kStream) == 1);
        t.borrow(theirs);
        EXPECT(t.create() == cudaSuccess && t.get() != theirs && live(kStream) == 2);
        t.borrow(theirs);
        EXPECT(live(kStream) == 1);
    }
    EXPECT(live(kStream) == 1 && g_live.count((uintptr_t)theirs));
    EXPECT(cudaStreamDestroy(theirs) == cudaSuccess && g_live.empty());
    return 0;
}

}  // extern "C"
