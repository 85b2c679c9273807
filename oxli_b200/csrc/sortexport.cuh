// sortexport.cuh -- device LSD radix sort of exported (hash, count) pairs.
//
// Stands in for the host sorts of KmerCountTable::dump (/root/reference/src/lib.rs:330-381):
// `sortkeys` orders by hash, `sortcounts` by (count, hash) (the tuple order of lines 353-355).
// Stable 8-bit passes, least significant digit first, so "by (count, hash)" is the hash sort
// followed by as many passes over the counts as the largest count has bytes.
//
// One pass = three kernels over tiles of kSortTile pairs:
//   radix_hist     per tile, how many pairs carry each digit              -> hist[digit][tile]
//   radix_scan     exclusive scan of hist in (digit, tile) order           -> where each tile's
//                                                                             digit run begins
//   radix_scatter  pairs to their places, order inside a (tile, digit) run preserved
// Stability inside a tile: the tile is walked in rounds of one pair per thread; within a round a
// pair's rank among equals is (equal digits in lower warps) + (equal digits in lower lanes),
// from one __match_any_sync per warp and a per-warp count table in shared memory.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace oxg {

constexpr int kSortThreads = 256;
constexpr int kSortRounds = 16;
constexpr int kSortTile = kSortThreads * kSortRounds;  // 4096 pairs per CTA

// Key mode (by_count == 0) also sorts keys alone: vals (and vals_out) == nullptr, and no value is
// loaded or stored.

// sort digit of pair i: bits [shift, shift+8) of the hash (by_count == 0) or of the count
__device__ __forceinline__ uint32_t sort_digit(const uint64_t *keys, const uint64_t *vals, uint64_t i, int shift, int by_count) {
    return (uint32_t)(((by_count ? vals[i] : keys[i]) >> shift) & 0xffu);
}

static __global__ void __launch_bounds__(kSortThreads) radix_hist_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ vals,
                                                                         uint64_t n, int shift, int by_count, uint64_t n_tiles,
                                                                         uint64_t *__restrict__ hist) {
    __shared__ uint32_t cnt[256];
    cnt[threadIdx.x] = 0;
    __syncthreads();
    const uint64_t base = (uint64_t)blockIdx.x * kSortTile;
    for (int r = 0; r < kSortRounds; ++r) {
        const uint64_t i = base + (uint64_t)r * kSortThreads + threadIdx.x;
        if (i < n) atomicAdd(&cnt[sort_digit(keys, vals, i, shift, by_count)], 1u);
    }
    __syncthreads();
    hist[(uint64_t)threadIdx.x * n_tiles + blockIdx.x] = cnt[threadIdx.x];
}

// exclusive scan of `m` counters in place (single CTA of 1024 threads)
static __global__ void __launch_bounds__(1024) radix_scan_kernel(uint64_t *__restrict__ a, uint64_t m) {
    __shared__ uint64_t part[1024];
    const uint64_t per = (m + blockDim.x - 1) / blockDim.x;
    const uint64_t lo = min(m, threadIdx.x * per), hi = min(m, lo + per);
    uint64_t s = 0;
    for (uint64_t i = lo; i < hi; ++i) s += a[i];
    part[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint64_t run = 0;
        for (uint32_t i = 0; i < blockDim.x; ++i) { const uint64_t v = part[i]; part[i] = run; run += v; }
    }
    __syncthreads();
    uint64_t run = part[threadIdx.x];
    for (uint64_t i = lo; i < hi; ++i) { const uint64_t v = a[i]; a[i] = run; run += v; }
}

static __global__ void __launch_bounds__(kSortThreads) radix_scatter_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ vals,
                                                                            uint64_t *__restrict__ keys_out, uint64_t *__restrict__ vals_out,
                                                                            uint64_t n, int shift, int by_count, uint64_t n_tiles,
                                                                            const uint64_t *__restrict__ offsets) {
    constexpr int kWarps = kSortThreads / 32;
    __shared__ uint32_t warp_cnt[kWarps][256];
    __shared__ uint64_t run_base[256];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    run_base[threadIdx.x] = offsets[(uint64_t)threadIdx.x * n_tiles + blockIdx.x];
    const uint64_t base = (uint64_t)blockIdx.x * kSortTile;
    for (int r = 0; r < kSortRounds; ++r) {
        for (int w = 0; w < kWarps; ++w) warp_cnt[w][threadIdx.x] = 0;
        __syncthreads();
        const uint64_t i = base + (uint64_t)r * kSortThreads + threadIdx.x;
        const bool valid = i < n;
        const uint64_t k = valid ? keys[i] : 0, v = valid && vals ? vals[i] : 0;
        const uint32_t d = valid ? (uint32_t)(((by_count ? v : k) >> shift) & 0xffu) : 0x100u + (uint32_t)lane;  // pairs past the end match nobody
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const uint32_t rank_in_warp = __popc(peers & ((1u << lane) - 1));
        if (valid && rank_in_warp == 0) warp_cnt[warp][d] = __popc(peers);
        __syncthreads();
        if (valid) {
            uint32_t before = 0;
            for (int w = 0; w < warp; ++w) before += warp_cnt[w][d];
            const uint64_t at = run_base[d] + before + rank_in_warp;
            keys_out[at] = k;
            if (vals_out) vals_out[at] = v;
        }
        __syncthreads();
        uint32_t tot = 0;
        for (int w = 0; w < kWarps; ++w) tot += warp_cnt[w][threadIdx.x];
        run_base[threadIdx.x] += tot;
        __syncthreads();
    }
}

}  // namespace oxg
