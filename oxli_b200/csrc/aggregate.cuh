// aggregate.cuh -- pass B of the partitioned counting pipeline.
//
// Together with consume_kernel<K, kModePart> (pass A) this replaces the per-window
// `count_hash` of KmerCountTable::consume (/root/reference/src/lib.rs:586-600, 100-104)
// by "scatter, pre-reduce duplicates, then update":
//
//   pass A   hashes the reads and scatters every hash into the fragment of its destination,
//            a destination being (owning rank, contiguous segment of that rank's table) --
//            the partition index is the top bits of h * phi, the same product whose top bits
//            are the slot index.
//   pass B   (this file) one CTA at a time takes a partition, streams its fragments -- from
//            every source rank: the pointers may be peer memory, then these loads are the
//            multi-GPU exchange -- through a shared-memory table that adds up duplicates
//            (key -> occurrences in this launch), and merges the distinct keys into the table
//            in HBM with one update each, in slot order.
//
// Why: a random 16-byte read-modify-write per k-mer is bound by L1TEX wavefronts and L2
// atomics at ~45 G k-mers/s on a hot table (profiles/r1_microbench_table_updates.txt).  After
// partitioning, all occurrences of a key inside a launch meet in one CTA: on high-coverage
// input (C2: every key ~10x per 64 M-window launch) nine of ten updates never leave shared
// memory, and what does reach the table walks one small segment in ascending slot order.
//
// The shared-memory table is a cache, not a container: a hash that finds its neighbourhood
// full (kLocalProbe buckets) bypasses it and updates the table in HBM directly, so a
// partition with more distinct keys than the cache holds (singleton-heavy input) degrades
// to the direct path without any mode switch, and skew is harmless: the spill list of pass A
// (a k-mer flooding its partition, e.g. poly-A) is cut into slices that any CTA aggregates.
#pragma once
#include "table.cuh"

namespace oxg {

constexpr int kAggThreadsDefault = 768;              // one CTA per SM; 85 registers per thread keep the
                                                     // prefetched block of hashes out of local memory
constexpr int kLocalBits = 14;
constexpr uint32_t kLocalSlots = 1u << kLocalBits;  // 16384 x (8-byte key + 4-byte count) = 192 KB
constexpr int kLocalProbe = 2;                      // buckets of four slots examined before bypassing
constexpr uint32_t kSpillSlice = 1u << 16;          // spill-list entries per work item
constexpr int kMaxSources = 16;
constexpr uint32_t kAggMaxFrags = 296 * kMaxSources;  // fragments of one partition: pass A CTAs (up to two per
                                                      // SM of a B200) x sources

struct AggSource {
    const uint64_t *frag;                 // [n_dest_total][n_ctas][frag_cap]
    const uint32_t *frag_cnt;             // [n_dest_total][n_ctas]
    const uint64_t *spill;
    const unsigned long long *spill_n;
};

struct AggParams {
    TableView table;
    AggSource src[kMaxSources];
    int n_src;
    uint32_t n_parts;     // partitions of THIS rank's table
    uint32_t dest0;       // self_rank * n_parts: first destination index that is ours
    uint32_t n_ctas;      // grid of pass A (fragments per destination and source)
    uint32_t frag_cap;
    uint32_t part_bits;   // log2(n_parts)
    uint32_t groups;      // work items per partition: item (part, g) takes the fragments f with f % groups == g
                          // (aggregate_groups: few with the cache on, some thousands of items in all with it off)
    uint32_t use_cache;   // 0: nothing to pre-reduce (nearly every key new): update the table directly
    uint64_t spill_cap;
    int owner_shift, self_rank, n_ranks;  // owner(h) = h >> owner_shift, for the spill lists
    unsigned long long *work_counter;     // zeroed before the launch
};

// ---- how many distinct keys will the table hold after this group of launches? ----------------
// HyperLogLog over the hashes pass A left in the fragments and the spill list (they are murmur
// outputs: the top kSketchBits bits pick the register, the rest give the rank), folded into the
// table's own sketch with max -- so the sketch estimates |keys of the table U keys of the group|
// and the table can be grown ONCE, before pass B, instead of running into its load limit,
// deferring, rehashing and replaying (an unhinted singleton-heavy stream ran at 0.4x the hinted
// rate that way).  2^13 registers (32 KB of shared memory per CTA): standard error 1.15 %.
constexpr int kSketchBits = 13;
constexpr uint32_t kSketchRegs = 1u << kSketchBits;

__global__ void __launch_bounds__(512) sketch_kernel(const AggParams p, uint32_t *__restrict__ sketch) {
    __shared__ uint32_t regs[kSketchRegs];
    for (uint32_t i = threadIdx.x; i < kSketchRegs; i += blockDim.x) regs[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
    auto see = [&](uint64_t h) {
        const uint32_t rho = (uint32_t)__clzll((long long)((h << kSketchBits) | (1ull << (kSketchBits - 1)))) + 1;
        atomicMax(&regs[h >> (64 - kSketchBits)], rho);
    };
    // fragments of this rank's partitions, one warp per fragment
    const uint64_t n_frag = (uint64_t)p.n_parts * p.n_ctas * (uint32_t)p.n_src;
    for (uint64_t f = (uint64_t)blockIdx.x * warps + warp; f < n_frag; f += (uint64_t)gridDim.x * warps) {
        const uint32_t part = (uint32_t)(f / (p.n_ctas * (uint32_t)p.n_src));
        const uint32_t rest = (uint32_t)(f % (p.n_ctas * (uint32_t)p.n_src));
        const uint32_t s = rest / p.n_ctas, c = rest % p.n_ctas;
        const uint64_t row = (uint64_t)(p.dest0 + part) * p.n_ctas + c;
        const uint32_t n = min(__ldg(p.src[s].frag_cnt + row), p.frag_cap);
        const uint64_t *ptr = p.src[s].frag + row * p.frag_cap;
        for (uint32_t i = lane; i < n; i += 32) {
            const uint64_t h = __ldcs(ptr + i);
            if (h != 0) see(h);
        }
    }
    for (int s = 0; s < p.n_src; ++s) {
        const uint64_t n = min((uint64_t)*p.src[s].spill_n, p.spill_cap);
        for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
            const uint64_t h = p.src[s].spill[i];
            if (p.n_ranks == 1 || (int)(h >> p.owner_shift) == p.self_rank) see(h);
        }
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < kSketchRegs; i += blockDim.x)
        if (regs[i]) atomicMax(&sketch[i], regs[i]);
}

inline size_t aggregate_smem_bytes(bool cache = true) { return (cache ? (size_t)kLocalSlots * 12 : 0) + (size_t)kAggMaxFrags * 4; }

// One occurrence of h into the shared-memory table.  false = neighbourhood full, bypass.
// Buckets of four slots (two 128-bit shared loads): at the loads this table runs at, a key sits in
// its home bucket 99 times out of 100, so the probe loop almost never takes a second, divergent
// turn (with two-slot buckets it did for one warp step in two, and pass B took 13.8 instead of
// 9.4 ms per C2 step at twice the load).  Slots only ever go from empty to a key, so a stale
// "empty" is caught by the CAS and a stale "other key" cannot happen; equal keys racing for a slot
// agree on it through the CAS result.  A key lives in the first bucket of its probe sequence that
// had a free slot when it came, and buckets never empty, so a lookup that walks past full buckets
// finds it.
__device__ __forceinline__ bool local_count(uint64_t *lk, uint32_t *ld, uint64_t h, uint32_t bucket) {
    uint32_t b = bucket << 2;
#pragma unroll 1
    for (int pr = 0; pr < kLocalProbe; ++pr) {
        const ulonglong2 k01 = *reinterpret_cast<const ulonglong2 *>(lk + b);
        const ulonglong2 k23 = *reinterpret_cast<const ulonglong2 *>(lk + b + 2);
        const uint64_t kk[4] = {k01.x, k01.y, k23.x, k23.y};
        int at = -1;
#pragma unroll
        for (int i = 3; i >= 0; --i) at = kk[i] == h ? i : at;
        if (at >= 0) { atomicAdd(ld + b + at, 1u); return true; }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (kk[i] != kEmpty) continue;
            const uint64_t old = atomicCAS((unsigned long long *)(lk + b + i), (unsigned long long)kEmpty, (unsigned long long)h);
            if (old == kEmpty || old == h) { atomicAdd(ld + b + i, 1u); return true; }
        }
        b = (b + 4) & (kLocalSlots - 1);
    }
    return false;
}

// kCache = false (p.use_cache == 0): no shared-memory table, every hash updates the table in HBM;
// the registers the cache path needs go to twice as many table loads in flight per lane (this
// variant is bound by the latency of those loads: 69 % of its stall samples are long-scoreboard,
// profiles/r2_aggregate_direct_ncu_summary.txt).
template <int kAggThreads, bool kCache>
__global__ void __launch_bounds__(kAggThreads, 1) aggregate_kernel(const AggParams p) {
    extern __shared__ __align__(16) uint8_t agg_smem[];
    uint64_t *lk = reinterpret_cast<uint64_t *>(agg_smem);                    // keys
    uint32_t *ld = reinterpret_cast<uint32_t *>(agg_smem + kLocalSlots * 8);  // occurrences
    uint32_t *s_end = kCache ? ld + kLocalSlots : reinterpret_cast<uint32_t *>(agg_smem);  // the item's fragments, where their hashes end
    __shared__ unsigned long long s_item;
    __shared__ uint32_t s_next;                          // next run of blocks past the ranges (or spill block) of the item
    __shared__ uint32_t s_blocks;                        // blocks of the item
    __shared__ uint32_t s_warp_sum[kAggThreads / 32];
    __shared__ uint64_t s_spill_first[kMaxSources + 1];  // work-item index of each source's first spill slice

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const TableView &tv = p.table;

    if (threadIdx.x == 0) {
        uint64_t run = (uint64_t)p.n_parts * p.groups;
        for (int s = 0; s < p.n_src; ++s) {
            s_spill_first[s] = run;
            const uint64_t n = min((uint64_t)*p.src[s].spill_n, p.spill_cap);
            run += (n + kSpillSlice - 1) / kSpillSlice;
        }
        s_spill_first[p.n_src] = run;
    }
    __syncthreads();
    const uint64_t n_items = s_spill_first[p.n_src];

    uint32_t created = 0;
    uint64_t n_taken = 0;  // occurrences this thread fed into the table (cache or direct)
    auto flush_created = [&]() {
        const uint32_t tot = __reduce_add_sync(0xffffffffu, created);
        if (lane == 0 && tot) atomicAdd((unsigned long long *)&tv.ctrl->size, (unsigned long long)tot);
        created = 0;
    };

    // U hashes per lane: through the shared-memory table first; what bypasses it goes to the
    // table in HBM with the home-bucket loads in flight together
    constexpr int U = 4;
    constexpr uint32_t kBlk = 32 * U;  // hashes a warp takes per step
    auto take = [&](const uint64_t (&h)[U], uint32_t live, bool full) {
        // (a straight-line "home buckets of all U first, probe loop for the rest" variant was
        // measured slower, 14.6 vs 9.4 ms per C2 step: the loop below already exits on its first
        // iteration nine times out of ten, and the variant loads every bucket twice on a miss)
        if constexpr (!kCache) {
            const uint64_t one[U] = {1, 1, 1, 1};
            if (live) created += table_add_many<U>(tv, h, one, live, full);
            return;
        }
        uint32_t direct = 0;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (!((live >> u) & 1u)) continue;
            const uint32_t bucket = (uint32_t)(((h[u] * kPhi) << p.part_bits) >> (64 - (kLocalBits - 2)));
            if (h[u] == kEmpty || !local_count(lk, ld, h[u], bucket)) direct |= 1u << u;
        }
        if (direct) {  // two at a time: four sets of bucket registers do not fit the register budget
            const uint64_t one[2] = {1, 1};
            const uint64_t lo2[2] = {h[0], h[1]}, hi2[2] = {h[2], h[3]};
            if (direct & 3u) created += table_add_many<2>(tv, lo2, one, direct & 3u, full);
            if (direct >> 2) created += table_add_many<2>(tv, hi2, one, direct >> 2, full);
        }
    };
    // the lanes' share of a block of n <= kBlk hashes at ptr
    auto load_blk = [&](const uint64_t *ptr, uint32_t n, uint64_t (&h)[U]) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t i = u * 32 + lane;
            h[u] = i < n ? __ldcs(ptr + i) : 0;
        }
    };
    auto take_blk = [&](const uint64_t (&h)[U], bool filter_owner, bool full) {
        uint32_t live = 0;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            bool ok = h[u] != 0;  // (0 fills the tail of a block past the fragment's fill count)
            if (filter_owner && p.n_ranks > 1 && ok) ok = (int)(h[u] >> p.owner_shift) == p.self_rank;
            live |= (ok ? 1u : 0u) << u;
        }
        n_taken += __popc(live);
        take(h, live, full);
    };

    for (;;) {
        __syncthreads();  // previous item fully merged; s_item free
        if (threadIdx.x == 0) { s_item = atomicAdd(p.work_counter, 1ULL); s_next = 0; }
        // empty the cache
        if (kCache) {
            for (uint32_t i = threadIdx.x; i < kLocalSlots / 2; i += kAggThreads)
                reinterpret_cast<ulonglong2 *>(lk)[i] = make_ulonglong2(kEmpty, kEmpty);
            for (uint32_t i = threadIdx.x; i < kLocalSlots / 4; i += kAggThreads)
                reinterpret_cast<uint4 *>(ld)[i] = make_uint4(0, 0, 0, 0);
        }
        __syncthreads();
        const uint64_t item = s_item;
        if (item >= n_items) break;
        const bool full = tv.overflow != nullptr && __ldcg(&tv.ctrl->size) >= tv.limit;

        if (item < (uint64_t)p.n_parts * p.groups) {
            // A partition of this rank's table: its fragments from every source and pass-A CTA
            // (with groups > 1, one share of them: fragments g, g + groups, ...).  Laid end to end,
            // each padded to whole blocks of kBlk hashes, they are the item's blocks; the warps take
            // them in that order, always one block ahead.  Only filled blocks are handed out: a fragment is planned for every window position of its share plus some
            // margin (plan_partitioned) and is typically half full.
            const uint64_t dest = p.dest0 + item / p.groups;
            const uint32_t g = (uint32_t)(item % p.groups);
            const uint32_t n_frag = min(p.n_ctas * (uint32_t)p.n_src, kAggMaxFrags);
            const uint32_t n_mine = g < n_frag ? (n_frag - g + p.groups - 1) / p.groups : 0;
            auto row_of = [&](uint32_t i, int &s) {  // fragment i of the item: its source and row
                const uint32_t f = g + i * p.groups;
                s = (int)(f / p.n_ctas);
                return dest * p.n_ctas + (f - (uint32_t)s * p.n_ctas);
            };
            // s_end[i] = where fragment i's hashes end in the item's blocks: kBlk x (blocks of the
            // fragments before it) + its fill count.  A scan over contiguous runs of fragments per
            // thread.  (Below 2^32: a partition's fragments from all sources hold at most half of
            // what one source's do, under 2^31 entries -- plan_partitioned -- and padding adds < kBlk
            // per fragment.)
            const uint32_t per = (n_mine + kAggThreads - 1) / kAggThreads;
            const uint32_t i0 = min(threadIdx.x * per, n_mine), i1 = min(i0 + per, n_mine);
            uint32_t mine = 0;
            for (uint32_t i = i0; i < i1; ++i) {
                int s;
                const uint64_t row = row_of(i, s);
                const uint32_t fill = min(__ldg(p.src[s].frag_cnt + row), p.frag_cap);
                s_end[i] = fill;
                mine += (fill + kBlk - 1) / kBlk * kBlk;
            }
            uint32_t before = mine;
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, before, o);
                if (lane >= o) before += y;
            }
            if (lane == 31) s_warp_sum[warp] = before;
            before -= mine;
            __syncthreads();
            if (warp == 0) {
                const uint32_t v = lane < kAggThreads / 32 ? s_warp_sum[lane] : 0u;
                uint32_t x = v;
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
                    if (lane >= o) x += y;
                }
                if (lane < kAggThreads / 32) s_warp_sum[lane] = x - v;
                if (lane == 31) s_blocks = x / kBlk;
            }
            __syncthreads();
            before += s_warp_sum[warp];
            for (uint32_t i = i0; i < i1; ++i) {
                const uint32_t fill = s_end[i];
                s_end[i] = before + fill;
                before += (fill + kBlk - 1) / kBlk * kBlk;
            }
            __syncthreads();
            const uint32_t n_blocks = s_blocks;
            // the fragment holding block blk: the first i with s_end[i] > blk * kBlk (the empty fragments
            // before it end where it starts), 32 candidates per step
            auto frag_of = [&](uint32_t blk) {
                const uint32_t x = blk * kBlk;
                uint32_t lo = 0, hi = n_mine - 1;  // it is in [lo, hi]
                while (lo < hi) {
                    const uint32_t step = (hi - lo + 32) / 32, at = lo + lane * step + step - 1;
                    lo += step * __popc(__ballot_sync(0xffffffffu, at < hi && s_end[at] <= x));
                    hi = min(hi, lo + step - 1);
                }
                return lo;
            };
            // The first seven eighths of the blocks are split evenly among the warps up front, one
            // contiguous range each; the rest is handed out in runs of a warp's share of what is left
            // (so that the last runs are short and the warps finish level).  A warp streams each
            // fragment of a range or run front to back.  Measured per step: runs from the first block
            // on took 8.42 ms of pass B on C2 against 8.11 (one block per run: 9.85), ranges over all
            // blocks 35.62 ms on C3-shaped input, whose small items of the cache-less variant need the
            // level finish, against 34.94.
            const uint32_t n_ranged = n_blocks - n_blocks / 8;
            uint32_t b = (uint32_t)((uint64_t)warp * n_ranged / (kAggThreads / 32));                // next block
            uint32_t b_end = (uint32_t)((uint64_t)(warp + 1) * n_ranged / (kAggThreads / 32));      // end of the range or run
            uint32_t left = 0;  // hashes of the fragment in hand, up to b_end
            const uint64_t *cur = nullptr;
            auto next_blk = [&](const uint64_t *&ptr, uint32_t &n) {  // warp-uniform; n = 0: nothing left
                if (!left) {
                    if (b >= b_end) {
                        uint32_t t = 0, run = 0;
                        if (lane == 0) {
                            const uint32_t seen = *(volatile uint32_t *)&s_next;
                            run = max(1u, (n_blocks - n_ranged - min(seen, n_blocks - n_ranged)) / (kAggThreads / 32));
                            t = n_ranged + atomicAdd(&s_next, run);
                        }
                        b = __shfl_sync(0xffffffffu, t, 0);
                        if (b >= n_blocks) { n = 0; return; }
                        b_end = min(b + __shfl_sync(0xffffffffu, run, 0), n_blocks);
                    }
                    const uint32_t j = frag_of(b);
                    const uint32_t first = j ? (s_end[j - 1] + kBlk - 1) / kBlk * kBlk : 0u;  // fragment j's first block, x kBlk
                    int s;
                    const uint64_t row = row_of(j, s);
                    cur = p.src[s].frag + row * p.frag_cap + (b * kBlk - first);
                    left = min(s_end[j], b_end * kBlk) - b * kBlk;
                }
                ptr = cur; n = min(left, kBlk);
                cur += n; left -= n; ++b;
            };
            const uint64_t *ptr = nullptr, *ptr2 = nullptr;
            uint32_t n = 0, n2 = 0;
            uint64_t h[U], h2[U];
            next_blk(ptr, n);
            if (n) load_blk(ptr, n, h);
            while (n) {
                next_blk(ptr2, n2);
                if (n2) load_blk(ptr2, n2, h2);
                take_blk(h, false, full);
                n = n2;
#pragma unroll
                for (int u = 0; u < U; ++u) h[u] = h2[u];
            }
            flush_created();
        } else {
            // a slice of some source's spill list (hashes of any partition, any owner)
            int s = 0;
            while (item >= s_spill_first[s + 1]) ++s;
            const uint64_t n_sp = min((uint64_t)*p.src[s].spill_n, p.spill_cap);
            const uint64_t lo = (item - s_spill_first[s]) * kSpillSlice;
            const uint64_t hi = min(n_sp, lo + kSpillSlice);
            for (;;) {
                uint32_t b = 0;
                if (lane == 0) b = atomicAdd(&s_next, 1u);
                b = __shfl_sync(0xffffffffu, b, 0);
                const uint64_t at = lo + (uint64_t)b * kBlk;
                if (at >= hi) break;
                uint64_t h[U];
                load_blk(p.src[s].spill + at, (uint32_t)min((uint64_t)kBlk, hi - at), h);
                take_blk(h, true, full);
            }
            flush_created();
        }
        __syncthreads();  // the cache holds every occurrence that did not bypass it

        // merge: distinct keys of this item, in slot order of the table (the cache index is the
        // next-lower bits of the same product h * phi)
        if (kCache) {
            constexpr int M = 2;
            for (uint32_t base = 0; base < kLocalSlots; base += kAggThreads * M) {
                uint64_t key[M], inc[M];
                uint32_t live = 0;
#pragma unroll
                for (int u = 0; u < M; ++u) {
                    const uint32_t i = base + u * kAggThreads + threadIdx.x;
                    key[u] = i < kLocalSlots ? lk[i] : kEmpty;
                    inc[u] = i < kLocalSlots ? ld[i] : 0u;
                    live |= (key[u] != kEmpty ? 1u : 0u) << u;
                }
                if (live) created += table_add_many<M>(tv, key, inc, live, full);
            }
            flush_created();
        }
    }
    for (int o = 16; o; o >>= 1) n_taken += __shfl_xor_sync(0xffffffffu, n_taken, o);
    if (lane == 0 && n_taken) atomicAdd((unsigned long long *)&tv.ctrl->absorbed, (unsigned long long)n_taken);
}

}  // namespace oxg
