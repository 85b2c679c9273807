// owned.h -- owners of the C ABI's CUDA resources: device arrays (plain or stream-ordered), pinned
// host arrays, events and streams.  Releases are quiet: they skip what is not held and clear any
// error their call reports, so that an error return keeps its message.
#pragma once
#include <algorithm>
#include <atomic>
#include <cassert>
#include <cstdint>
#include <utility>
#include <cuda_runtime.h>

namespace oxg {

// resources held by owners now, and the countdown to an allocation that fails as out of memory
// (0: none), for tests of the error returns (oxg_live_allocations, oxg_fail_allocation_after)
inline std::atomic<uint64_t> g_owned_live{0}, g_owned_fail_in{0};

// every allocation and handle creation of an owner: make() unless the countdown ends here
template <class Make>
cudaError_t owned_acquire(Make &&make) {
    uint64_t n = g_owned_fail_in.load();
    while (n && !g_owned_fail_in.compare_exchange_weak(n, n - 1)) {}
    const cudaError_t e = n == 1 ? cudaErrorMemoryAllocation : make();
    if (e != cudaSuccess) cudaGetLastError();
    else g_owned_live.fetch_add(1);
    return e;
}
inline void owned_release(cudaError_t e) {
    if (e != cudaSuccess) cudaGetLastError();
    g_owned_live.fetch_sub(1);
}

// Move-only T[cap] in device memory -- cudaMalloc / cudaFree, or, given a stream (which must outlive
// the array), cudaMallocAsync / cudaFreeAsync on it -- or in pinned host memory; with a grow-only
// reserve that does not keep the old contents.  A failed reserve leaves the owner empty.
template <class T, bool Pinned>
class OwnedArray {
public:
    OwnedArray() = default;
    explicit OwnedArray(cudaStream_t ordered_on) : st_(ordered_on) { assert(ordered_on); }
    OwnedArray(OwnedArray &&o) noexcept { *this = std::move(o); }
    OwnedArray &operator=(OwnedArray &&o) noexcept {
        if (this != &o) { reset(); std::swap(p_, o.p_); std::swap(cap_, o.cap_); std::swap(st_, o.st_); }
        return *this;
    }
    ~OwnedArray() { reset(); }
    T *get() const { return p_; }
    uint64_t cap() const { return cap_; }
    // from now on freed onto stream st (an array from cudaMalloc that is to go without a device sync)
    void free_on(cudaStream_t st) { assert(st); st_ = st; }
    // room for n entries, min_cap at least (nothing when both are 0)
    cudaError_t reserve(uint64_t n, uint64_t min_cap = 0) {
        const uint64_t want = std::max(n, min_cap), bytes = want * sizeof(T);
        if (cap_ >= n && (p_ || want == 0)) return cudaSuccess;
        reset();
        void *q = nullptr;
        const cudaError_t e = owned_acquire([&] {
            return Pinned ? cudaMallocHost(&q, bytes) : st_ ? cudaMallocAsync(&q, bytes, st_) : cudaMalloc(&q, bytes);
        });
        if (e == cudaSuccess) { p_ = static_cast<T *>(q); cap_ = want; }
        return e;
    }
    void reset() {
        if (p_) owned_release(Pinned ? cudaFreeHost(p_) : st_ ? cudaFreeAsync(p_, st_) : cudaFree(p_));
        p_ = nullptr; cap_ = 0;
    }
private:
    T *p_ = nullptr;
    uint64_t cap_ = 0;
    cudaStream_t st_ = nullptr;
};
template <class T> using DeviceArray = OwnedArray<T, false>;
template <class T> using PinnedArray = OwnedArray<T, true>;

// a stream drains before it goes: the stream-ordered frees queued on it, and its copies out of
// buffers released after it
inline cudaError_t drain_and_destroy(cudaStream_t s) {
    const cudaError_t e = cudaStreamSynchronize(s), d = cudaStreamDestroy(s);
    return e != cudaSuccess ? e : d;
}

// an event or stream handle (neither copied nor moved), created with flags; it converts to H for
// the calls that take one
template <class H, cudaError_t (*Create)(H *, unsigned), cudaError_t (*Destroy)(H)>
class OwnedHandle {
public:
    OwnedHandle() = default;
    OwnedHandle(const OwnedHandle &) = delete;
    OwnedHandle &operator=(const OwnedHandle &) = delete;
    ~OwnedHandle() { reset(); }
    operator H() const { return h_; }
    cudaError_t create(unsigned flags) {
        reset();
        const cudaError_t e = owned_acquire([&] { return Create(&h_, flags); });
        if (e != cudaSuccess) h_ = nullptr;
        return e;
    }
    void reset() { if (h_) owned_release(Destroy(h_)); h_ = nullptr; }
private:
    H h_ = nullptr;
};
using Event = OwnedHandle<cudaEvent_t, cudaEventCreateWithFlags, cudaEventDestroy>;
using Stream = OwnedHandle<cudaStream_t, cudaStreamCreateWithFlags, drain_and_destroy>;

}  // namespace oxg
