// dump.cuh -- text of sorted (hash, count) pairs: the reference's dump lines "<hash>\t<count>\n"
// (src/lib.rs:330-381; u64 in decimal, as pyoxli.cpp's dump prints them), 4 to 42 bytes a line.
//
// Pairs are taken in tiles of kDumpTile; a CTA owns one tile.
//   dump_length_kernel   bytes of each tile's text                     -> tile_off[tile]
//   (radix_scan_kernel)  exclusive scan of tile_off (one extra entry)  -> where each tile's text begins
//   dump_bounds_kernel   byte position of given pair positions (the run boundaries of a rank's export)
//   dump_format_kernel   each tile's text, staged in shared memory, stored to its place with 16-byte
//                        stores (bytes only at the two ends of a tile)
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace oxg {

constexpr int kDumpThreads = 256;
constexpr int kDumpPer = 4;                           // consecutive pairs per thread
constexpr int kDumpTile = kDumpThreads * kDumpPer;    // 1024 pairs per CTA
constexpr int kDumpLineMax = 20 + 1 + 20 + 1;

// decimal digits of x (1 for 0)
__device__ __forceinline__ uint32_t dec_digits(uint64_t x) {
    uint32_t d = 1;
    uint64_t p = 10;
#pragma unroll
    for (int i = 1; i < 20; ++i, p *= 10) d += x >= p ? 1u : 0u;
    return d;
}

__device__ __forceinline__ uint32_t dump_line_bytes(uint64_t k, uint64_t v) { return dec_digits(k) + dec_digits(v) + 2; }

// x in decimal, `digits` bytes ending just before `end`, two digits at a time from the table
__device__ __forceinline__ void put_dec(uint8_t *end, uint64_t x, const uint8_t *__restrict__ tab) {
    while (x >= 100) {
        const uint64_t q = x / 100;
        const uint32_t r = (uint32_t)(x - q * 100);
        end -= 2;
        end[0] = tab[2 * r]; end[1] = tab[2 * r + 1];
        x = q;
    }
    if (x >= 10) { end -= 2; end[0] = tab[2 * x]; end[1] = tab[2 * x + 1]; }
    else *--end = (uint8_t)('0' + x);
}

// exclusive prefix of v over the CTA (kDumpThreads threads); *total = the sum
__device__ __forceinline__ uint32_t dump_block_scan(uint32_t v, uint32_t *warp_tot, uint32_t *total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += y;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    uint32_t before = 0, all = 0;
#pragma unroll
    for (int w = 0; w < kDumpThreads / 32; ++w) {
        const uint32_t t = warp_tot[w];
        before += w < warp ? t : 0;
        all += t;
    }
    *total = all;
    return before + incl - v;
}

static __global__ void __launch_bounds__(kDumpThreads) dump_length_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ vals,
                                                                          uint64_t n, uint64_t *__restrict__ tile_off) {
    __shared__ uint32_t warp_tot[kDumpThreads / 32];
    const uint64_t i0 = (uint64_t)blockIdx.x * kDumpTile + threadIdx.x * kDumpPer;
    uint32_t mine = 0;
#pragma unroll
    for (int j = 0; j < kDumpPer; ++j)
        if (i0 + j < n) mine += dump_line_bytes(keys[i0 + j], vals[i0 + j]);
    uint32_t total;
    dump_block_scan(mine, warp_tot, &total);
    if (threadIdx.x == 0) tile_off[blockIdx.x] = total;
}

// pos[j] (a pair position in [0, n]) -> the byte position where its line begins (n: the end of the
// text), in place; tile_off scanned.  One warp per position, which sums the lines before it in its tile.
static __global__ void dump_bounds_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ vals,
                                          const uint64_t *__restrict__ tile_off, uint64_t *__restrict__ pos, uint64_t m) {
    const uint64_t j = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (j >= m) return;
    const uint64_t p = pos[j], t = p / kDumpTile;
    uint64_t sum = 0;
    for (uint64_t i = t * kDumpTile + lane; i < p; i += 32) sum += dump_line_bytes(keys[i], vals[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) pos[j] = tile_off[t] + sum;
}

// text of tiles [tile0, tile0 + gridDim.x) into out, which holds the text from tile0's first byte on
// and is 16-byte aligned
static __global__ void __launch_bounds__(kDumpThreads) dump_format_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ vals,
                                                                          uint64_t n, uint64_t tile0, const uint64_t *__restrict__ tile_off,
                                                                          uint8_t *__restrict__ out) {
    __shared__ __align__(16) uint8_t text[kDumpTile * kDumpLineMax + 16];
    __shared__ uint8_t tab[200];
    __shared__ uint32_t warp_tot[kDumpThreads / 32];
    if (threadIdx.x < 100) { tab[2 * threadIdx.x] = (uint8_t)('0' + threadIdx.x / 10); tab[2 * threadIdx.x + 1] = (uint8_t)('0' + threadIdx.x % 10); }
    const uint64_t tile = tile0 + blockIdx.x;
    const uint64_t i0 = tile * kDumpTile + threadIdx.x * kDumpPer;
    uint64_t k[kDumpPer], v[kDumpPer];
    uint32_t kd[kDumpPer], vd[kDumpPer], mine = 0;
#pragma unroll
    for (int j = 0; j < kDumpPer; ++j) {
        const bool ok = i0 + j < n;
        k[j] = ok ? keys[i0 + j] : 0; v[j] = ok ? vals[i0 + j] : 0;
        kd[j] = ok ? dec_digits(k[j]) : 0; vd[j] = ok ? dec_digits(v[j]) : 0;
        mine += ok ? kd[j] + vd[j] + 2 : 0;
    }
    uint32_t total;
    const uint32_t before = dump_block_scan(mine, warp_tot, &total);  // (its barrier also publishes tab)
    const uint64_t at = tile_off[tile] - tile_off[tile0];  // where this tile's text goes in out
    const uint32_t lead = (uint32_t)(at & 15);             // text[lead + x] is stored at out[at + x]
    uint8_t *p = text + lead + before;
#pragma unroll
    for (int j = 0; j < kDumpPer; ++j) {
        if (i0 + j >= n) break;
        put_dec(p + kd[j], k[j], tab);
        p[kd[j]] = '\t';
        p += kd[j] + 1;
        put_dec(p + vd[j], v[j], tab);
        p[vd[j]] = '\n';
        p += vd[j] + 1;
    }
    __syncthreads();
    // 16-byte words of out that the tile touches; the first and the last may be shared with the
    // neighbouring tiles, so only this tile's bytes of them are stored
    uint8_t *dst = out + (at - lead);
    const uint32_t end = lead + total, words = (end + 15) / 16;
    for (uint32_t w = threadIdx.x; w < words; w += kDumpThreads) {
        const uint32_t lo = 16 * w, hi = lo + 16;
        if (lo >= lead && hi <= end) {
            reinterpret_cast<uint4 *>(dst)[w] = reinterpret_cast<const uint4 *>(text)[w];
        } else {
            for (uint32_t b = max(lo, lead); b < min(hi, end); ++b) dst[b] = text[b];
        }
    }
}

}  // namespace oxg
