// lookup.cuh -- device side of the sharded table's lookup round (oxg_shard_get_hashes*).
//
// A round: every rank sorts its queries by owner into the fragment region of its own exchange
// area (route_*), each owner reads its segment of every rank's queries through the peer mapping,
// looks the keys up in its table and writes each count over its key (answer_queries_kernel), and
// every rank reads its answers back in the order of its queries (gather_answers_kernel).  Each key
// slot is read and rewritten by exactly one owner, so the answers need no memory of their own.
#pragma once
#include "shard.cuh"
#include "tableops.cuh"

namespace oxg {

constexpr int kRouteThreads = 256;
constexpr int kRouteWarps = kRouteThreads / 32;
constexpr int kRouteU = 4;  // queries per thread and tile: four loads in flight
constexpr int kRouteTile = kRouteU * kRouteThreads;
constexpr int kRouteScanThreads = 1024;

// owner(h) = h >> (64 - log2 N); owner_shift is 64 for one rank
__device__ __forceinline__ uint32_t owner_bin(uint64_t h, uint32_t owner_shift) {
    return owner_shift >= 64 ? 0u : (uint32_t)(h >> owner_shift);
}

// Route, step 1.  CTA c takes the queries [c * chunk, (c + 1) * chunk) of the round and counts
// them per owner in shared memory: bins[o * gridDim.x + c] (one shared atomic per warp and owner).
__global__ void __launch_bounds__(kRouteThreads) route_count_kernel(const uint64_t *__restrict__ q, uint64_t m, uint64_t chunk,
                                                                    uint32_t owner_shift, uint32_t n_own, uint32_t *__restrict__ bins) {
    __shared__ uint32_t hist[kShardMaxRanks];
    if (threadIdx.x < kShardMaxRanks) hist[threadIdx.x] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint64_t lo = min(m, blockIdx.x * chunk), hi = min(m, lo + chunk);
    for (uint64_t t0 = lo; t0 < hi; t0 += kRouteTile) {
        uint32_t o[kRouteU];
#pragma unroll
        for (int u = 0; u < kRouteU; ++u) {
            const uint64_t i = t0 + u * kRouteThreads + threadIdx.x;
            o[u] = i < hi ? owner_bin(q[i], owner_shift) : kShardMaxRanks;
        }
#pragma unroll
        for (int u = 0; u < kRouteU; ++u) {
            const uint32_t peers = __match_any_sync(0xffffffffu, o[u]);
            if (o[u] < kShardMaxRanks && lane == __ffs(peers) - 1) atomicAdd(&hist[o[u]], __popc(peers));
        }
    }
    __syncthreads();
    if (threadIdx.x < n_own) bins[threadIdx.x * gridDim.x + blockIdx.x] = hist[threadIdx.x];
}

// Route, step 2 (one CTA of kRouteScanThreads).  bins becomes its exclusive prefix sum in (owner,
// CTA) order: the slot where CTA c's run of owner o begins.  offs[o] = first slot of owner o's
// segment, offs[n_own] = m.
__global__ void __launch_bounds__(kRouteScanThreads) route_scan_kernel(uint32_t *__restrict__ bins, uint32_t n_bins, uint32_t grid,
                                                                       uint32_t n_own, uint64_t m, uint64_t *__restrict__ offs) {
    __shared__ uint32_t warp_sum_s[kRouteScanThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t per = (n_bins + kRouteScanThreads - 1) / kRouteScanThreads;
    const uint32_t b0 = min(n_bins, threadIdx.x * per), b1 = min(n_bins, b0 + per);
    uint32_t mine = 0;
    for (uint32_t i = b0; i < b1; ++i) mine += bins[i];
    uint32_t inc = mine;  // inclusive scan over the warp
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += v;
    }
    if (lane == 31) warp_sum_s[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const uint32_t w = warp_sum_s[lane];
        uint32_t wi = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, wi, d);
            if (lane >= d) wi += v;
        }
        warp_sum_s[lane] = wi - w;
    }
    __syncthreads();
    uint32_t run = warp_sum_s[warp] + inc - mine;
    for (uint32_t i = b0; i < b1; ++i) {
        const uint32_t v = bins[i];
        bins[i] = run;
        run += v;
    }
    __syncthreads();
    if (threadIdx.x <= n_own) offs[threadIdx.x] = threadIdx.x < n_own ? bins[threadIdx.x * grid] : m;
}

// Route, step 3: the same chunks as step 1, tile by tile in index order.  Each query goes to the
// next slot of its owner's run in frag (stable: slots follow the queries' order), and pos[i]
// records where.  A tile writes at most one contiguous run per owner.
__global__ void __launch_bounds__(kRouteThreads) route_queries_kernel(const uint64_t *__restrict__ q, uint64_t m, uint64_t chunk,
                                                                      uint32_t owner_shift, uint32_t n_own,
                                                                      const uint32_t *__restrict__ base, uint64_t *__restrict__ frag,
                                                                      uint32_t *__restrict__ pos) {
    constexpr int kVW = kRouteU * kRouteWarps;              // (u, warp): 32 queries each, in index order
    __shared__ uint32_t cnt[kVW][kShardMaxRanks];           // queries per (u, warp) and owner
    __shared__ uint32_t first[kVW][kShardMaxRanks];         // ... and the slot of the first of them
    __shared__ uint32_t next[kShardMaxRanks];               // this CTA's next free slot per owner
    for (int j = threadIdx.x; j < kVW * kShardMaxRanks; j += kRouteThreads) (&cnt[0][0])[j] = 0;
    if (threadIdx.x < n_own) next[threadIdx.x] = base[threadIdx.x * gridDim.x + blockIdx.x];
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t below = (1u << lane) - 1;
    const uint64_t lo = min(m, blockIdx.x * chunk), hi = min(m, lo + chunk);
    for (uint64_t t0 = lo; t0 < hi; t0 += kRouteTile) {
        uint64_t h[kRouteU];
        uint32_t o[kRouteU], peers[kRouteU];
#pragma unroll
        for (int u = 0; u < kRouteU; ++u) {
            const uint64_t i = t0 + u * kRouteThreads + threadIdx.x;
            h[u] = i < hi ? q[i] : 0;
            o[u] = i < hi ? owner_bin(h[u], owner_shift) : kShardMaxRanks;
        }
#pragma unroll
        for (int u = 0; u < kRouteU; ++u) {
            peers[u] = __match_any_sync(0xffffffffu, o[u]);
            if (o[u] < kShardMaxRanks && lane == __ffs(peers[u]) - 1) cnt[u * kRouteWarps + warp][o[u]] = __popc(peers[u]);
        }
        __syncthreads();
        if (threadIdx.x < n_own) {
            uint32_t run = next[threadIdx.x];
            for (int v = 0; v < kVW; ++v) {
                first[v][threadIdx.x] = run;
                run += cnt[v][threadIdx.x];
                cnt[v][threadIdx.x] = 0;
            }
            next[threadIdx.x] = run;
        }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < kRouteU; ++u) {
            if (o[u] >= kShardMaxRanks) continue;
            const uint32_t at = first[u * kRouteWarps + warp][o[u]] + __popc(peers[u] & below);
            frag[at] = h[u];
            pos[t0 + u * kRouteThreads + threadIdx.x] = at;
        }
    }
}

// Where the owner finds every rank's queries of the round: rank s's routed queries (frag) and
// its n + 1 owner offsets (offs), both through the peer mapping.
struct LookupSources {
    uint64_t *frag[kShardMaxRanks];
    const uint64_t *offs[kShardMaxRanks];
    int n;
};

// On the owner `me`: the segments [offs_s[me], offs_s[me + 1]) of every rank s, concatenated into
// one grid-stride range.  Four keys per thread are loaded (coalesced, over NVLink for a peer's)
// before table_get_many looks them up; each count is one 8-byte store over its key.
__global__ void __launch_bounds__(kOpThreads) answer_queries_kernel(TableView t, LookupSources src, int me) {
    __shared__ uint64_t seg_lo[kShardMaxRanks];       // segment s starts at this slot of rank s's frag
    __shared__ uint64_t seg_at[kShardMaxRanks + 1];   // ... and at this position of the concatenation
    if ((int)threadIdx.x < src.n) {
        const uint64_t lo = __ldcg(src.offs[threadIdx.x] + me), hi = __ldcg(src.offs[threadIdx.x] + me + 1);
        seg_lo[threadIdx.x] = lo;
        seg_at[threadIdx.x + 1] = hi - lo;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        seg_at[0] = 0;
        for (int s = 1; s <= src.n; ++s) seg_at[s] += seg_at[s - 1];
    }
    __syncthreads();
    constexpr int U = 4;
    const uint64_t total = seg_at[src.n], stride = gstride();
    for (uint64_t base = gtid(); base < total; base += stride * U) {
        uint64_t *p[U], key[U], cnt[U];
        uint32_t live = 0;
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const uint64_t i = base + j * stride;
            p[j] = nullptr;
            key[j] = 0;
            if (i < total) {
                int s = 0;
                while (i >= seg_at[s + 1]) ++s;
                p[j] = src.frag[s] + seg_lo[s] + (i - seg_at[s]);
                key[j] = __ldcg(p[j]);
                live |= 1u << j;
            }
        }
        table_get_many<U>(t, key, live, cnt);
#pragma unroll
        for (int j = 0; j < U; ++j)
            if ((live >> j) & 1) *p[j] = cnt[j];
    }
}

// out[i] = frag[pos[i]]: this rank's answers, back in the order of its queries
__global__ void __launch_bounds__(kOpThreads) gather_answers_kernel(const uint64_t *frag, const uint32_t *__restrict__ pos, uint64_t m,
                                                                    uint64_t *__restrict__ out) {
    for (uint64_t i = gtid(); i < m; i += gstride()) out[i] = __ldcg(frag + pos[i]);
}

}  // namespace oxg
