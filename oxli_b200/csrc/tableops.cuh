// tableops.cuh -- table maintenance, lookup, reduction, export and set kernels.
// Each kernel names the reference method it stands in for
// (paths: /root/reference/src/lib.rs).
#pragma once
#include "table.cuh"

namespace oxg {

constexpr int kOpThreads = 256;
constexpr uint32_t kHistSmem = 1024;    // counts below this: per-CTA shared bins
constexpr uint32_t kHistDense = 65536;  // counts below this: dense global bins; above: listed raw
constexpr int kExportChunk = 4096;      // slots per CTA in the ordered export

__device__ __forceinline__ uint64_t gtid() { return blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; }
__device__ __forceinline__ uint64_t gstride() { return gridDim.x * (uint64_t)blockDim.x; }

__device__ __forceinline__ uint64_t warp_sum(uint64_t v) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// HashMap::new / clear
__global__ void init_slots_kernel(ulonglong2 *slots, uint64_t cap) {
    for (uint64_t i = gtid(); i < cap; i += gstride()) slots[i] = make_ulonglong2(kEmpty, 0);
}

// count_hash for a list (src/lib.rs:100-104); room was reserved by the host.
// Without new_counts: 4 keys per thread per round (8 was slower: scripts/microbench_probe.cu), all home buckets (one 256-bit
// load each) requested before the first is examined; zero keys are skipped when
// skip_zero is set (the hash stream of the two-kernel pipeline marks bad windows 0).
__global__ void __launch_bounds__(kOpThreads) count_hashes_kernel(TableView t, const uint64_t *__restrict__ hashes, uint64_t n,
                                    uint64_t *__restrict__ new_counts, int skip_zero) {
    uint32_t created = 0;
    uint64_t counted = 0;
    if (new_counts) {
        for (uint64_t i = gtid(); i < n; i += gstride())
            new_counts[i] = table_add_fetch(t, hashes[i], 1, &created);
    } else {
        constexpr int U = 4;
        const uint64_t stride = gstride();
        for (uint64_t base = gtid(); base < n; base += stride * U) {
            // at the load limit new keys are deferred to the overflow list (if there is one)
            const bool full = t.overflow != nullptr && __ldcg(&t.ctrl->size) >= t.limit;
            uint64_t h[U], idx[U];
            ulonglong2 a[U], b[U];
            bool live[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint64_t i = base + u * stride;
                live[u] = i < n;
                h[u] = live[u] ? __ldcs(hashes + i) : 0;
                if (skip_zero && h[u] == 0) live[u] = false;
                if (h[u] == kEmpty) { if (live[u]) { created += table_add(t, h[u], 1, full); ++counted; } live[u] = false; }
                idx[u] = t.home(h[u]);
            }
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (live[u]) load_pair(t.slots + idx[u], a[u], b[u]);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (!live[u]) continue;
                ++counted;
                if (a[u].x == h[u]) red_add64(&t.slots[idx[u]].y, 1);
                else if (b[u].x == h[u]) red_add64(&t.slots[idx[u] + 1].y, 1);
                else {
                    const bool redo = a[u].x == kEmpty || b[u].x == kEmpty;
                    created += table_add_buckets(t, h[u], 1, full, (idx[u] + (redo ? 0 : 2)) & (t.cap - 1));
                }
            }
        }
    }
    const uint64_t tot = warp_sum(created);
    counted = warp_sum(counted);
    if ((threadIdx.x & 31) == 0) {
        if (tot) atomicAdd((unsigned long long *)&t.ctrl->size, (unsigned long long)tot);
        if (counted) atomicAdd((unsigned long long *)&t.ctrl->counted, (unsigned long long)counted);
    }
}

// Replay of a deferral list: counts[key] += inc for (key, inc) pairs, four in flight per thread;
// at the load limit again, pairs go on to the view's own deferral list.
__global__ void __launch_bounds__(kOpThreads) replay_pairs_kernel(TableView t, const ulonglong2 *__restrict__ pairs, uint64_t n) {
    constexpr int U = 4;
    uint32_t created = 0;
    const uint64_t stride = gstride();
    for (uint64_t base = gtid(); base < n; base += stride * U) {
        const bool full = t.overflow != nullptr && __ldcg(&t.ctrl->size) >= t.limit;
        uint64_t key[U], inc[U];
        uint32_t live = 0;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint64_t i = base + u * stride;
            const ulonglong2 e = i < n ? pairs[i] : make_ulonglong2(0, 0);
            key[u] = e.x; inc[u] = e.y;
            live |= (i < n ? 1u : 0u) << u;
        }
        created += table_add_many<U>(t, key, inc, live, full);
    }
    const uint64_t tot = warp_sum(created);
    if ((threadIdx.x & 31) == 0 && tot) atomicAdd((unsigned long long *)&t.ctrl->size, (unsigned long long)tot);
}

// counts[key] += val for (key,val) pairs; creates keys (also with val == 0)
__global__ void add_pairs_kernel(TableView t, const uint64_t *__restrict__ keys, const uint64_t *__restrict__ vals, uint64_t n) {
    uint32_t created = 0;
    for (uint64_t i = gtid(); i < n; i += gstride()) created += table_add(t, keys[i], vals[i], false);
    const uint64_t tot = warp_sum(created);
    if ((threadIdx.x & 31) == 0 && tot) atomicAdd((unsigned long long *)&t.ctrl->size, (unsigned long long)tot);
}

// get_hash / get_hash_array (src/lib.rs:185-194)
__global__ void get_hashes_kernel(TableView t, const uint64_t *__restrict__ hashes, uint64_t n,
                                  uint64_t *__restrict__ out) {
    constexpr int U = 4;
    const uint64_t stride = gstride();
    for (uint64_t base = gtid(); base < n; base += stride * U) {
        uint64_t key[U], cnt[U];
        uint32_t live = 0;
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const uint64_t i = base + j * stride;
            key[j] = i < n ? hashes[i] : 0;
            live |= (i < n ? 1u : 0u) << j;
        }
        table_get_many<U>(t, key, live, cnt);
#pragma unroll
        for (int j = 0; j < U; ++j)
            if ((live >> j) & 1) out[base + j * stride] = cnt[j];
    }
}

// __setitem__: counts.insert(hash, value) (src/lib.rs:675-681).  One thread.
__global__ void set_hash_kernel(TableView t, uint64_t key, uint64_t value) {
    if (gtid() != 0) return;
    if (key == kEmpty) { t.ctrl->side_present = 1; t.ctrl->side_count = value; return; }
    uint64_t i = t.home(key);
    for (;;) {
        ulonglong2 s = t.slots[i];
        if (s.x == key) { t.slots[i].y = value; return; }
        if (s.x == kEmpty) { t.slots[i] = make_ulonglong2(key, value); t.ctrl->size += 1; return; }
        i = (i + 1) & (t.cap - 1);
    }
}

// drop_hash of one key (src/lib.rs:213-224): remove it, then shift the rest of the probe run back
// so lookups never need tombstones; 2^64-1 clears the side entry.  ++removed when the key was
// there.  Only one thread of the grid may erase at a time.
__device__ __forceinline__ void erase_one(const TableView &t, uint64_t key, uint64_t &removed) {
    if (key == kEmpty) {
        if (t.ctrl->side_present) { t.ctrl->side_present = 0; t.ctrl->side_count = 0; ++removed; }
        return;
    }
    int64_t f = table_find(t, key);
    if (f < 0) return;
    const uint64_t mask = t.cap - 1;
    uint64_t hole = (uint64_t)f, j = hole;
    t.slots[hole] = make_ulonglong2(kEmpty, 0);
    for (;;) {
        j = (j + 1) & mask;
        ulonglong2 s = t.slots[j];
        if (s.x == kEmpty) break;
        const uint64_t hm = t.home(s.x);
        // s may move into the hole iff its home is not cyclically inside (hole, j]
        if (((j - hm) & mask) >= ((j - hole) & mask)) {
            t.slots[hole] = s;
            t.slots[j] = make_ulonglong2(kEmpty, 0);
            hole = j;
        }
    }
    ++removed;
    t.ctrl->size -= 1;
}

// drop_hash for a short list: one thread walks it.
__global__ void erase_hashes_kernel(TableView t, const uint64_t *__restrict__ hashes, uint64_t n) {
    if (gtid() != 0) return;
    uint64_t removed = 0;
    for (uint64_t q = 0; q < n; ++q) erase_one(t, hashes[q], removed);
    t.ctrl->scratch[0] = removed;
}

// Marks the slot of `key` (not 2^64-1) in a bitmap of one bit per slot; ++found when this call set
// the bit, so a key listed twice counts once.
__device__ __forceinline__ void erase_mark_one(const TableView &t, uint64_t key, uint32_t *__restrict__ doomed, uint64_t &found) {
    const int64_t f = table_find(t, key);
    if (f < 0) return;
    const uint32_t bit = 1u << (f & 31);
    if (!(atomicOr(&doomed[f >> 5], bit) & bit)) ++found;
}

// Bulk form of drop_hash: mark the slots of the listed keys in a bitmap (one bit per slot; a key
// listed twice is marked once), then rebuild without them (erase_rebuild_kernel) -- the
// single-thread kernel above is for the reference's one-key calls, this one for lists.
// scratch[0] += keys found.
__global__ void erase_mark_kernel(TableView t, const uint64_t *__restrict__ hashes, uint64_t n, uint32_t *__restrict__ doomed) {
    uint64_t found = 0;
    for (uint64_t q = gtid(); q < n; q += gstride()) {
        const uint64_t key = hashes[q];
        if (key == kEmpty) continue;  // the out-of-band key is handled on the host
        erase_mark_one(t, key, doomed, found);
    }
    found = warp_sum(found);
    if ((threadIdx.x & 31) == 0 && found) atomicAdd((unsigned long long *)&t.ctrl->scratch[0], (unsigned long long)found);
}

__global__ void erase_rebuild_kernel(const ulonglong2 *__restrict__ old_slots, uint64_t old_cap, TableView nt, const uint32_t *__restrict__ doomed) {
    for (uint64_t i = gtid(); i < old_cap; i += gstride()) {
        const ulonglong2 s = old_slots[i];
        if (s.x == kEmpty || ((doomed[i >> 5] >> (i & 31)) & 1u)) continue;
        table_add(nt, s.x, s.y, false);
    }
}

// growth: re-insert every live entry of the old slot array
__global__ void rehash_kernel(const ulonglong2 *__restrict__ old_slots, uint64_t old_cap, TableView nt) {
    for (uint64_t i = gtid(); i < old_cap; i += gstride()) {
        ulonglong2 s = old_slots[i];
        if (s.x != kEmpty) table_add(nt, s.x, s.y, false);
    }
}

// mincut / maxcut (src/lib.rs:227-267): rebuild keeping the survivors.
// mode 0 drops count < thresh, mode 1 drops count > thresh.
__global__ void cut_kernel(const ulonglong2 *__restrict__ old_slots, uint64_t old_cap, TableView nt,
                           int mode, uint64_t thresh) {
    uint64_t removed = 0;
    for (uint64_t i = gtid(); i < old_cap; i += gstride()) {
        ulonglong2 s = old_slots[i];
        if (s.x == kEmpty) continue;
        const bool drop = mode == 0 ? (s.y < thresh) : (s.y > thresh);
        if (drop) ++removed; else table_add(nt, s.x, s.y, false);
    }
    removed = warp_sum(removed);
    if ((threadIdx.x & 31) == 0 && removed) atomicAdd((unsigned long long *)&nt.ctrl->scratch[0], (unsigned long long)removed);
}

// __len__, sum_counts, min, max and histo in one pass (src/lib.rs:464-539, 665).
// scratch: [0]=len [1]=sum [2]=min [3]=max [4]=number of raw (>= kHistDense) values
__global__ void stats_kernel(TableView t, uint64_t *__restrict__ dense, uint64_t *__restrict__ big,
                             uint64_t big_cap) {
    __shared__ uint32_t bins[kHistSmem];
    for (uint32_t i = threadIdx.x; i < kHistSmem; i += blockDim.x) bins[i] = 0;
    __syncthreads();
    uint64_t len = 0, sum = 0, mn = ~0ULL, mx = 0;
    for (uint64_t i = gtid(); i < t.cap; i += gstride()) {
        ulonglong2 s = t.slots[i];
        if (s.x == kEmpty) continue;
        const uint64_t v = s.y;
        ++len; sum += v; mn = min(mn, v); mx = max(mx, v);
        if (dense) {
            if (v < kHistSmem) atomicAdd(&bins[v], 1u);
            else if (v < kHistDense) atomicAdd((unsigned long long *)&dense[v], 1ULL);
            else {
                uint64_t at = atomicAdd((unsigned long long *)&t.ctrl->scratch[4], 1ULL);
                if (at < big_cap) big[at] = v;
            }
        }
    }
    len = warp_sum(len); sum = warp_sum(sum);
    for (int o = 16; o; o >>= 1) {
        mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if ((threadIdx.x & 31) == 0 && len) {
        atomicAdd((unsigned long long *)&t.ctrl->scratch[0], (unsigned long long)len);
        atomicAdd((unsigned long long *)&t.ctrl->scratch[1], (unsigned long long)sum);
        atomicMin((unsigned long long *)&t.ctrl->scratch[2], (unsigned long long)mn);
        atomicMax((unsigned long long *)&t.ctrl->scratch[3], (unsigned long long)mx);
    }
    __syncthreads();
    if (dense)
        for (uint32_t i = threadIdx.x; i < kHistSmem; i += blockDim.x)
            if (bins[i]) atomicAdd((unsigned long long *)&dense[i], (unsigned long long)bins[i]);
}

// Order-independent digests of the (key, count) multiset, for parity checks at sizes where
// nothing can be exported: scratch [0]=len [1]=sum c [2]=xor h [3]=sum h*c (wrapping)
// [4]=keys whose owner (h >> owner_shift) differs from `rank` (owner_shift 64: not sharded).
__global__ void digest_kernel(TableView t, int owner_shift, uint64_t rank) {
    uint64_t len = 0, sum = 0, x = 0, hc = 0, foreign = 0;
    for (uint64_t i = gtid(); i < t.cap; i += gstride()) {
        const ulonglong2 s = t.slots[i];
        if (s.x == kEmpty) continue;
        ++len; sum += s.y; x ^= s.x; hc += s.x * s.y;
        if (owner_shift < 64 && (s.x >> owner_shift) != rank) ++foreign;
    }
    len = warp_sum(len); sum = warp_sum(sum); hc = warp_sum(hc); foreign = warp_sum(foreign);
    for (int o = 16; o; o >>= 1) x ^= __shfl_xor_sync(0xffffffffu, x, o);
    if ((threadIdx.x & 31) == 0 && len) {
        atomicAdd((unsigned long long *)&t.ctrl->scratch[0], (unsigned long long)len);
        atomicAdd((unsigned long long *)&t.ctrl->scratch[1], (unsigned long long)sum);
        atomicXor((unsigned long long *)&t.ctrl->scratch[2], (unsigned long long)x);
        atomicAdd((unsigned long long *)&t.ctrl->scratch[3], (unsigned long long)hc);
        if (foreign) atomicAdd((unsigned long long *)&t.ctrl->scratch[4], (unsigned long long)foreign);
    }
}

// ---- ordered export: hashes / dump / __iter__ (src/lib.rs:330-381, 517-521, 658-662)
// pass 1: live slots per chunk of kExportChunk slots
__global__ void export_count_kernel(const ulonglong2 *__restrict__ slots, uint64_t cap,
                                    uint64_t *__restrict__ chunk_counts) {
    __shared__ uint32_t total;
    if (threadIdx.x == 0) total = 0;
    __syncthreads();
    const uint64_t base = blockIdx.x * (uint64_t)kExportChunk;
    uint32_t c = 0;
    for (uint32_t i = threadIdx.x; i < kExportChunk; i += blockDim.x)
        if (base + i < cap && slots[base + i].x != kEmpty) ++c;
    c = (uint32_t)warp_sum(c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&total, c);
    __syncthreads();
    if (threadIdx.x == 0) chunk_counts[blockIdx.x] = total;
}

// exclusive scan of chunk_counts in place (single CTA); total -> *out_total
__global__ void export_scan_kernel(uint64_t *__restrict__ chunk_counts, uint64_t n, uint64_t *out_total) {
    __shared__ uint64_t part[1024];
    const uint64_t per = (n + blockDim.x - 1) / blockDim.x;
    const uint64_t lo = min(n, threadIdx.x * per), hi = min(n, lo + per);
    uint64_t s = 0;
    for (uint64_t i = lo; i < hi; ++i) s += chunk_counts[i];
    part[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint64_t run = 0;
        for (uint32_t i = 0; i < blockDim.x; ++i) { uint64_t v = part[i]; part[i] = run; run += v; }
        *out_total = run;
    }
    __syncthreads();
    uint64_t run = part[threadIdx.x];
    for (uint64_t i = lo; i < hi; ++i) { uint64_t v = chunk_counts[i]; chunk_counts[i] = run; run += v; }
}

// pass 2: write (key,count) of live slots in slot order
__global__ void export_write_kernel(const ulonglong2 *__restrict__ slots, uint64_t cap,
                                    const uint64_t *__restrict__ chunk_offsets,
                                    uint64_t *__restrict__ keys, uint64_t *__restrict__ vals,
                                    uint64_t out_cap) {
    constexpr int PER = kExportChunk / kOpThreads;  // consecutive slots per thread
    __shared__ uint32_t pre[kOpThreads];
    const uint64_t base = blockIdx.x * (uint64_t)kExportChunk + threadIdx.x * (uint64_t)PER;
    ulonglong2 s[PER];
    uint32_t c = 0;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        s[i] = base + i < cap ? slots[base + i] : make_ulonglong2(kEmpty, 0);
        c += s[i].x != kEmpty;
    }
    pre[threadIdx.x] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t run = 0;
        for (int i = 0; i < kOpThreads; ++i) { uint32_t v = pre[i]; pre[i] = run; run += v; }
    }
    __syncthreads();
    uint64_t at = chunk_offsets[blockIdx.x] + pre[threadIdx.x];
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        if (s[i].x == kEmpty) continue;
        if (at < out_cap) { keys[at] = s[i].x; if (vals) vals[at] = s[i].y; }
        ++at;
    }
}

// ---- set comparisons (src/lib.rs:610-638, 708-722): |A & B| by probing B with A's keys
__global__ void setop_count_kernel(TableView a, TableView b) {
    constexpr int U = 4;
    uint64_t both = 0;
    const uint64_t stride = gstride();
    for (uint64_t base = gtid(); base < a.cap; base += stride * U) {
        uint64_t key[U], cnt[U];
        uint32_t live = 0;
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const uint64_t i = base + j * stride;
            key[j] = i < a.cap ? __ldcs(&a.slots[i].x) : kEmpty;
            live |= (key[j] != kEmpty ? 1u : 0u) << j;
        }
        if (live) both += __popc(table_get_many<U>(b, key, live, cnt));
    }
    both = warp_sum(both);
    if ((threadIdx.x & 31) == 0 && both) atomicAdd((unsigned long long *)&a.ctrl->scratch[0], (unsigned long long)both);
}

// keys of A whose membership in B equals want_in_b (2 = don't care); unordered append
__global__ void setop_export_kernel(TableView a, TableView b, int want_in_b, uint64_t *__restrict__ out,
                                    uint64_t out_cap, uint64_t *out_count) {
    const uint64_t n = (a.cap + 31) / 32 * 32;  // keep warps whole for the ballots
    for (uint64_t i = gtid(); i < n; i += gstride()) {
        const uint64_t k = i < a.cap ? a.slots[i].x : kEmpty;
        bool emit = k != kEmpty;
        if (emit && want_in_b != 2) emit = (table_find(b, k) >= 0) == (want_in_b == 1);
        const unsigned m = __ballot_sync(0xffffffffu, emit);
        if (!m) continue;
        const int lane = threadIdx.x & 31;
        uint64_t base = 0;
        if (lane == 0) base = atomicAdd((unsigned long long *)out_count, (unsigned long long)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        const uint64_t at = base + __popc(m & ((1u << lane) - 1));
        if (emit && at < out_cap) out[at] = k;
    }
}

// cosine (src/lib.rs:727-765): scratch[0] = sum_{k in A&B} a_k*b_k (wrapping u64),
// scratch_f64[0] += sum a_k^2 as doubles
__global__ void cosine_kernel(TableView a, TableView b, double *__restrict__ sumsq_a) {
    uint64_t dot = 0;
    double sq = 0.0;
    constexpr int U = 4;
    const uint64_t stride = gstride();
    for (uint64_t base = gtid(); base < a.cap; base += stride * U) {
        uint64_t key[U], mine[U], cnt[U];
        uint32_t live = 0;
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const uint64_t i = base + j * stride;
            const ulonglong2 s = i < a.cap ? a.slots[i] : make_ulonglong2(kEmpty, 0);
            key[j] = s.x; mine[j] = s.y;
            live |= (s.x != kEmpty ? 1u : 0u) << j;
        }
        if (!live) continue;
#pragma unroll
        for (int j = 0; j < U; ++j)
            if ((live >> j) & 1) sq += (double)mine[j] * (double)mine[j];
        if (b.slots) {
            table_get_many<U>(b, key, live, cnt);
#pragma unroll
            for (int j = 0; j < U; ++j) dot += mine[j] * cnt[j];
        }
    }
    dot = warp_sum(dot);
    for (int o = 16; o; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    if ((threadIdx.x & 31) == 0) {
        if (dot) atomicAdd((unsigned long long *)&a.ctrl->scratch[0], (unsigned long long)dot);
        if (sq != 0.0) atomicAdd(sumsq_a, sq);
    }
}

// add (src/lib.rs:778-837): dst[k] += src[k]; scratch[0] = counts added,
// scratch[1] = keys whose previous count was 0 (the reference's "new keys")
__global__ void merge_kernel(TableView dst, TableView src) {
    uint64_t added = 0, fresh = 0;
    uint32_t created = 0;
    for (uint64_t i = gtid(); i < src.cap; i += gstride()) {
        ulonglong2 s = src.slots[i];
        if (s.x == kEmpty) continue;
        const uint64_t after = table_add_fetch(dst, s.x, s.y, &created);
        if (after - s.y == 0) ++fresh;
        added += s.y;
    }
    added = warp_sum(added); fresh = warp_sum(fresh);
    const uint64_t cr = warp_sum(created);
    if ((threadIdx.x & 31) == 0) {
        if (added) atomicAdd((unsigned long long *)&dst.ctrl->scratch[0], (unsigned long long)added);
        if (fresh) atomicAdd((unsigned long long *)&dst.ctrl->scratch[1], (unsigned long long)fresh);
        if (cr) atomicAdd((unsigned long long *)&dst.ctrl->size, (unsigned long long)cr);
    }
}

// ---- synthetic reads (SURVEY.md 8d): counter-based, reproducible on the CPU ----
__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}

__host__ __device__ __forceinline__ uint32_t genome_base(uint64_t seed, uint64_t pos) {
    return (uint32_t)(splitmix64(seed + (pos >> 5)) >> (2 * (pos & 31))) & 3u;  // 0..3 = A,C,G,T
}

__global__ void synth_reads_kernel(uint8_t *__restrict__ out, uint64_t n_reads, uint32_t read_len,
                                   uint64_t genome_len, uint64_t seed, uint64_t first_read,
                                   uint32_t sub_ppm, uint32_t n_ppm) {
    const uint64_t total = n_reads * read_len;
    for (uint64_t i = gtid(); i < total; i += gstride()) {
        const uint64_t r = i / read_len;
        const uint32_t j = (uint32_t)(i - r * read_len);
        const uint64_t rk = splitmix64((seed ^ 0x5EEDF00DULL) + (first_read + r) * 0x2545F4914F6CDD1DULL);
        const uint64_t start = rk % (genome_len - read_len + 1);
        const bool rev = (splitmix64(rk + 1) & 1) != 0;
        uint32_t b = rev ? 3u - genome_base(seed, start + read_len - 1 - j) : genome_base(seed, start + j);
        const uint64_t e = splitmix64(rk + 2 + j);
        if ((uint32_t)(e % 1000000u) < sub_ppm) b = (b + 1 + (uint32_t)((e >> 32) % 3u)) & 3u;
        uint8_t c = (uint8_t)"ACGT"[b];
        if ((uint32_t)((e >> 20) % 1000000u) < n_ppm) c = 'N';
        out[i] = c;
    }
}

}  // namespace oxg
