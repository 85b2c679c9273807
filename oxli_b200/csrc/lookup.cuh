// lookup.cuh -- device side of the sharded table's lookup, merge and erase rounds
// (oxg_shard_get_hashes*, oxg_shard_merge_table, oxg_shard_erase_hashes*).
//
// A lookup round: every rank sorts its queries by owner into the fragment region of its own
// exchange area (route_*), each owner reads its segment of every rank's queries through the peer
// mapping, looks the keys up in its table and writes each count over its key
// (answer_queries_kernel), and every rank reads its answers back in the order of its queries
// (gather_answers_kernel).  Each key slot is read and rewritten by exactly one owner, so the
// answers need no memory of their own.
//
// A merge round routes the occupied slots of a range of a plain table instead: keys to the
// fragment region, their counts to the same positions of the spill region, and each owner adds
// its segments into its table (apply_pairs_kernel).
//
// An erase round routes a list of keys as a lookup does, and each owner erases its segments from
// its table: in place for a few keys (erase_walk_segments_kernel), or by marking their slots for
// one rebuild after the last round (erase_mark_segments_kernel).
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

// Where a route's keys come from.  A list of queries (lookups): every entry is a key, and
// out[i] = the slot query i went to (pos) ...
struct RouteList {
    using In = uint64_t;
    using Out = uint32_t;
    static __device__ __forceinline__ uint64_t key(const In *q, uint64_t i) { return q[i]; }
    static __device__ __forceinline__ bool live(uint64_t) { return true; }
    static __device__ __forceinline__ uint32_t bin(const In *q, uint64_t i, uint32_t owner_shift) { return owner_bin(q[i], owner_shift); }
    static __device__ __forceinline__ void place(const In *, uint64_t i, uint32_t at, Out *out) { out[i] = at; }
};
// ... or a range of table slots (merges): empty slots go nowhere (so the out-of-band key never
// travels), and each key's count goes to the same position of out (the spill region) as the key
// goes to in frag.
struct RouteSlots {
    using In = ulonglong2;
    using Out = uint64_t;
    static __device__ __forceinline__ uint64_t key(const In *q, uint64_t i) { return q[i].x; }
    static __device__ __forceinline__ bool live(uint64_t h) { return h != kEmpty; }
    static __device__ __forceinline__ uint32_t bin(const In *q, uint64_t i, uint32_t owner_shift) {
        const uint64_t h = key(q, i);
        return live(h) ? owner_bin(h, owner_shift) : kShardMaxRanks;
    }
    static __device__ __forceinline__ void place(const In *q, uint64_t i, uint32_t at, Out *out) { out[at] = q[i].y; }
};

// Route, step 1.  CTA c takes the entries [c * chunk, (c + 1) * chunk) of the round and counts
// the keys among them per owner in shared memory: bins[o * gridDim.x + c] (one shared atomic per
// warp and owner).
template <class Src>
__global__ void __launch_bounds__(kRouteThreads) route_count_kernel(const typename Src::In *__restrict__ q, uint64_t m, uint64_t chunk,
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
            o[u] = i < hi ? Src::bin(q, i, owner_shift) : kShardMaxRanks;
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
// segment, offs[n_own] = the keys routed (the last thread's run ends at the total).
__global__ void __launch_bounds__(kRouteScanThreads) route_scan_kernel(uint32_t *__restrict__ bins, uint32_t n_bins, uint32_t grid,
                                                                       uint32_t n_own, uint64_t *__restrict__ offs) {
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
    if (threadIdx.x < n_own) offs[threadIdx.x] = bins[threadIdx.x * grid];
    if (threadIdx.x == kRouteScanThreads - 1) offs[n_own] = run;
}

// Route, step 3: the same chunks as step 1, tile by tile in index order.  Each key goes to the
// next slot of its owner's run in frag (stable: slots follow the entries' order), and Src::place
// records where (a query's slot) or what (a count) in out.  A tile writes at most one contiguous
// run per owner.
template <class Src>
__global__ void __launch_bounds__(kRouteThreads) route_queries_kernel(const typename Src::In *__restrict__ q, uint64_t m, uint64_t chunk,
                                                                      uint32_t owner_shift, uint32_t n_own,
                                                                      const uint32_t *__restrict__ base, uint64_t *__restrict__ frag,
                                                                      typename Src::Out *__restrict__ out) {
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
            h[u] = i < hi ? Src::key(q, i) : 0;
            o[u] = i < hi && Src::live(h[u]) ? owner_bin(h[u], owner_shift) : kShardMaxRanks;
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
            Src::place(q, t0 + u * kRouteThreads + threadIdx.x, at, out);
        }
    }
}

// Where the owner finds every rank's keys of the round: rank s's routed keys (frag) and its
// n + 1 owner offsets (offs), both through the peer mapping.
struct LookupSources {
    uint64_t *frag[kShardMaxRanks];
    const uint64_t *offs[kShardMaxRanks];
    int n;
};

// On the owner `me`: the segments [offs_s[me], offs_s[me + 1]) of every rank s, concatenated into
// one range.  seg_lo[s] = where segment s starts in rank s's region, seg_at[s] = where it starts in
// the concatenation (both in shared memory).  Called by every thread of the block (it
// synchronises); returns the range's length.
__device__ __forceinline__ uint64_t load_segments(const LookupSources &src, int me, uint64_t *seg_lo, uint64_t *seg_at) {
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
    return seg_at[src.n];
}

// entry i of that range: position `at` of rank `s`'s region
struct SegEntry { int s; uint64_t at; };
__device__ __forceinline__ SegEntry entry_of(const uint64_t *seg_lo, const uint64_t *seg_at, uint64_t i) {
    int s = 0;
    while (i >= seg_at[s + 1]) ++s;
    return SegEntry{s, seg_lo[s] + (i - seg_at[s])};
}

// Answers every rank's queries of the round: four keys per thread are loaded (coalesced, over
// NVLink for a peer's) before table_get_many looks them up; each count is one 8-byte store over
// its key.
__global__ void __launch_bounds__(kOpThreads) answer_queries_kernel(TableView t, LookupSources src, int me) {
    __shared__ uint64_t seg_lo[kShardMaxRanks], seg_at[kShardMaxRanks + 1];
    constexpr int U = 4;
    const uint64_t total = load_segments(src, me, seg_lo, seg_at), stride = gstride();
    for (uint64_t base = gtid(); base < total; base += stride * U) {
        uint64_t *p[U], key[U], cnt[U];
        uint32_t live = 0;
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const uint64_t i = base + j * stride;
            p[j] = nullptr;
            key[j] = 0;
            if (i < total) {
                const SegEntry e = entry_of(seg_lo, seg_at, i);
                p[j] = src.frag[e.s] + e.at;
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

// A merge round's routed pairs: the keys as a lookup's, and rank s's counts at the same positions
// of its spill region (vals[s]).
struct PairSources {
    LookupSources keys;
    const uint64_t *vals[kShardMaxRanks];
};

// On the owner `me`: counts[key] += count for every pair of every rank's segment (KmerCountTable::add,
// src/lib.rs:778-837), four in flight per thread.  Room for every key was reserved before the
// round (no deferral).  scratch[0] += counts added, scratch[1] += pairs whose key held 0 just
// before them (the reference's "new keys"), size += keys created; one atomic per warp each.
__global__ void __launch_bounds__(kOpThreads) apply_pairs_kernel(TableView t, PairSources src, int me) {
    __shared__ uint64_t seg_lo[kShardMaxRanks], seg_at[kShardMaxRanks + 1];
    constexpr int U = 4;
    const uint64_t total = load_segments(src.keys, me, seg_lo, seg_at), stride = gstride();
    uint64_t added = 0, fresh = 0;
    uint32_t created = 0;
    for (uint64_t base = gtid(); base < total; base += stride * U) {
        uint64_t key[U], val[U], before[U];
        uint32_t live = 0;
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const uint64_t i = base + j * stride;
            key[j] = 0;
            val[j] = 0;
            if (i < total) {
                const SegEntry e = entry_of(seg_lo, seg_at, i);
                key[j] = __ldcg(src.keys.frag[e.s] + e.at);
                val[j] = __ldcg(src.vals[e.s] + e.at);
                live |= 1u << j;
            }
        }
        created += table_add_fetch_many<U>(t, key, val, live, before);
#pragma unroll
        for (int j = 0; j < U; ++j)
            if ((live >> j) & 1) {
                added += val[j];
                fresh += before[j] == 0 ? 1 : 0;
            }
    }
    added = warp_sum(added);
    fresh = warp_sum(fresh);
    const uint64_t cr = warp_sum(created);
    if ((threadIdx.x & 31) == 0) {
        if (added) atomicAdd((unsigned long long *)&t.ctrl->scratch[0], (unsigned long long)added);
        if (fresh) atomicAdd((unsigned long long *)&t.ctrl->scratch[1], (unsigned long long)fresh);
        if (cr) atomicAdd((unsigned long long *)&t.ctrl->size, (unsigned long long)cr);
    }
}

// On the owner `me`, for a few keys over all ranks (drop / drop_hash, src/lib.rs:197-224): erase
// every key of every rank's segment in place, one at a time, as erase_hashes_kernel does -- no
// rebuild, so a single drop_hash costs a probe run, not a pass over the table.
// scratch[0] += keys removed, 2^64-1 included.  One thread walks; the block loads the segments.
__global__ void __launch_bounds__(32) erase_walk_segments_kernel(TableView t, LookupSources src, int me) {
    __shared__ uint64_t seg_lo[kShardMaxRanks], seg_at[kShardMaxRanks + 1];
    const uint64_t total = load_segments(src, me, seg_lo, seg_at);
    if (gtid() != 0) return;
    uint64_t removed = 0;
    for (uint64_t i = 0; i < total; ++i) {
        const SegEntry e = entry_of(seg_lo, seg_at, i);
        erase_one(t, __ldcg(src.frag[e.s] + e.at), removed);
    }
    t.ctrl->scratch[0] += removed;
}

// On the owner `me`, for a list: mark the slot of every key of every rank's segment in doomed (one
// bit per slot of my table), four keys in flight per thread; the table is rebuilt without them
// after the call's last round (erase_rebuild_kernel), so nothing may move it in between.
// scratch[0] += bits newly set (a key listed several times, by any ranks, counts once);
// scratch[1] = 1 when 2^64-1 is listed (its side entry is dropped on the host, with the rebuild).
__global__ void __launch_bounds__(kOpThreads) erase_mark_segments_kernel(TableView t, LookupSources src, int me,
                                                                         uint32_t *__restrict__ doomed) {
    __shared__ uint64_t seg_lo[kShardMaxRanks], seg_at[kShardMaxRanks + 1];
    constexpr int U = 4;
    const uint64_t total = load_segments(src, me, seg_lo, seg_at), stride = gstride();
    uint64_t found = 0;
    bool side = false;
    for (uint64_t base = gtid(); base < total; base += stride * U) {
        uint64_t key[U];
        uint32_t live = 0;
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const uint64_t i = base + j * stride;
            key[j] = 0;
            if (i < total) {
                const SegEntry e = entry_of(seg_lo, seg_at, i);
                key[j] = __ldcg(src.frag[e.s] + e.at);
                live |= 1u << j;
            }
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            if (!((live >> j) & 1)) continue;
            if (key[j] == kEmpty) side = true;
            else erase_mark_one(t, key[j], doomed, found);
        }
    }
    found = warp_sum(found);
    if ((threadIdx.x & 31) == 0 && found) atomicAdd((unsigned long long *)&t.ctrl->scratch[0], (unsigned long long)found);
    if (side) t.ctrl->scratch[1] = 1;
}

}  // namespace oxg
