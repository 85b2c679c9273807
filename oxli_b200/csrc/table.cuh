// table.cuh -- open-addressing u64 -> u64 count table in HBM.
//
// Stands in for the reference's `counts: HashMap<u64,u64>`
// (/root/reference/src/lib.rs:33; entry/insert/get at 100-104, 178, 187, 679).
// Layout: `cap` (power of two) 16-byte slots {key, count}, linear probing from
// home(key) = ((key * phi64) >> (64 - log2 cap)) & ~1, i.e. from the first slot of
// a 32-byte, two-slot bucket.  An empty slot holds kEmpty as
// key; that one key value is kept outside the slot array (side_*), so every
// u64 -- including 0 and 2^64-1 -- is a legal key and 0 a legal count.
// No tombstones: single-key erase shifts the probe run back, bulk cuts rebuild.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace oxg {

constexpr uint64_t kEmpty = ~0ULL;
constexpr uint64_t kPhi = 0x9E3779B97F4A7C15ULL;
constexpr int kMaxProbe = 1024;

struct Ctrl {              // lives in device memory, mirrored to pinned host memory
    // line 0: table state, read by every warp (size) -- kept apart from the hot atomics
    uint64_t size;         // live keys in slots[]
    uint64_t side_present; // key kEmpty is present
    uint64_t side_count;   // its count
    uint64_t first_bad;    // error-mode scan: smallest bad window start
    uint64_t pad0[12];
    // line 1: per-launch counters (zeroed together before every consume launch)
    uint64_t counted;      // k-mers counted by the running consume launch
    uint64_t overflow;     // entries appended to the overflow list
    uint64_t absorbed;     // received hashes counted by the running launch
    uint64_t late_new;     // keys created by the last quarter of the launch's tiles (growth look-ahead)
    uint64_t pad1[12];
    // lines 2 and 3: the two work counters every warp hits with atomics
    uint64_t tile_counter;   // dynamic tile scheduler of the running consume launch
    uint64_t pad2[15];
    uint64_t absorb_counter; // same, for blocks of received hashes (sharded route launches)
    uint64_t pad3[15];
    uint64_t scratch[16];  // per-op outputs (stats, set sizes, ...)
};
static_assert(offsetof(Ctrl, counted) == 128 && offsetof(Ctrl, tile_counter) == 256 &&
              offsetof(Ctrl, absorb_counter) == 384 && offsetof(Ctrl, scratch) == 512, "Ctrl layout");

struct TableView {
    ulonglong2 *slots;
    uint64_t cap;      // power of two
    uint32_t shift;    // 64 - log2(cap)
    uint64_t limit;    // stop creating keys once size reaches this
    Ctrl *ctrl;
    ulonglong2 *overflow;  // deferred (key, increment) pairs (table too full), may be null
    uint64_t overflow_cap;
    // home slot: even, so a key's first two candidate slots share one 32-byte sector
    __device__ __forceinline__ uint64_t home(uint64_t key) const {
        return ((key * kPhi) >> shift) & ~1ULL;
    }
};

__device__ __forceinline__ void red_add64(unsigned long long *p, uint64_t v) {
    asm volatile("red.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__device__ __forceinline__ ulonglong2 load_slot(const ulonglong2 *p) { return __ldcg(p); }

// both slots of a home bucket with one 256-bit load (sm_100: LDG.E.256)
__device__ __forceinline__ void load_pair(const ulonglong2 *p, ulonglong2 &a, ulonglong2 &b) {
    asm("ld.global.cg.v4.u64 {%0,%1,%2,%3}, [%4];"
        : "=l"(a.x), "=l"(a.y), "=l"(b.x), "=l"(b.y)
        : "l"(p));
}

// Deferred updates go to one list of (key, increment) pairs with one cursor: the lanes that
// arrive together reserve their entries with a single atomic (a launch that fills the table
// defers tens of millions of hashes; one atomic each on one address cost 7x the kernel time).
__device__ __forceinline__ void push_overflow(const TableView &t, uint64_t key, uint64_t inc) {
    const unsigned peers = __activemask();
    const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd((unsigned long long *)&t.ctrl->overflow, (unsigned long long)__popc(peers));
    base = __shfl_sync(peers, base, leader);
    const uint64_t at = base + __popc(peers & ((1u << lane) - 1));
    if (t.overflow && at < t.overflow_cap) t.overflow[at] = make_ulonglong2(key, inc);
}

// counts[key] += inc.  `full` = do not create keys (the table reached its load
// limit): misses are deferred to the overflow list and replayed after growth.
// Returns 1 when a new key was created.
__device__ __forceinline__ uint32_t table_add(const TableView &t, uint64_t key, uint64_t inc,
                                              bool full) {
    if (key == kEmpty) {
        atomicAdd((unsigned long long *)&t.ctrl->side_count, (unsigned long long)inc);
        t.ctrl->side_present = 1;
        return 0;
    }
    uint64_t i = t.home(key);
    // only launches that carry a deferral list may give up on a long probe run
    for (int probe = 0; t.overflow == nullptr || probe < kMaxProbe; ++probe) {
        ulonglong2 s = load_slot(t.slots + i);
        if (s.x == key) {
            red_add64(&t.slots[i].y, inc);
            return 0;
        }
        if (s.x == kEmpty) {
            if (full) break;
            uint64_t old = atomicCAS((unsigned long long *)&t.slots[i].x, kEmpty, key);
            if (old == kEmpty) {
                red_add64(&t.slots[i].y, inc);
                return 1;
            }
            if (old == key) {
                red_add64(&t.slots[i].y, inc);
                return 0;
            }
        }
        i = (i + 1) & (t.cap - 1);
    }
    push_overflow(t, key, inc);
    return 0;
}

// Bucket-wise variant used to drain the consume kernels' slow queue: walks 32-byte
// buckets (two slots per 256-bit load) starting at even slot `i`, which the caller
// guarantees is not past the key's position (home, or home+2 when the home bucket
// was seen full of other keys).
__device__ __forceinline__ uint32_t table_add_buckets(const TableView &t, uint64_t key, uint64_t inc,
                                                      bool full, uint64_t i) {
    for (int probe = 0; t.overflow == nullptr || probe < kMaxProbe; probe += 2) {
        ulonglong2 s[2];
        load_pair(t.slots + i, s[0], s[1]);
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            if (s[q].x == key) {
                red_add64(&t.slots[i + q].y, inc);
                return 0;
            }
            if (s[q].x == kEmpty) {
                if (full) { push_overflow(t, key, inc); return 0; }
                const uint64_t old = atomicCAS((unsigned long long *)&t.slots[i + q].x, kEmpty, key);
                if (old == kEmpty || old == key) {
                    red_add64(&t.slots[i + q].y, inc);
                    return old == kEmpty ? 1u : 0u;
                }
            }
        }
        i = (i + 2) & (t.cap - 1);
    }
    push_overflow(t, key, inc);
    return 0;
}

// counts[key[u]] += inc[u] for the lanes' U live entries, all home buckets requested before the
// first is examined (one dependent random sector per update is what bounds this; see
// table_get_many).  Returns the number of keys created.
template <int U>
__device__ __forceinline__ uint32_t table_add_many(const TableView &t, const uint64_t (&key)[U], const uint64_t (&inc)[U],
                                                   uint32_t live, bool full) {
    uint64_t idx[U];
    ulonglong2 a[U], b[U];
    uint32_t created = 0;
#pragma unroll
    for (int u = 0; u < U; ++u) {
        if (((live >> u) & 1u) && key[u] == kEmpty) { created += table_add(t, key[u], inc[u], full); live &= ~(1u << u); }
        idx[u] = t.home(key[u]);
        if ((live >> u) & 1u) load_pair(t.slots + idx[u], a[u], b[u]);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        if (!((live >> u) & 1u)) continue;
        if (a[u].x == key[u]) red_add64(&t.slots[idx[u]].y, inc[u]);
        else if (b[u].x == key[u]) red_add64(&t.slots[idx[u] + 1].y, inc[u]);
        else {
            const bool redo = a[u].x == kEmpty || b[u].x == kEmpty;
            created += table_add_buckets(t, key[u], inc[u], full, (idx[u] + (redo ? 0 : 2)) & (t.cap - 1));
        }
    }
    return created;
}

// same, but returns the count after the increment (count_hash, src/lib.rs:100-104);
// never defers: the caller reserved room.
__device__ __forceinline__ uint64_t table_add_fetch(const TableView &t, uint64_t key, uint64_t inc,
                                                    uint32_t *created) {
    if (key == kEmpty) {
        t.ctrl->side_present = 1;
        return atomicAdd((unsigned long long *)&t.ctrl->side_count, (unsigned long long)inc) + inc;
    }
    uint64_t i = t.home(key);
    for (;;) {
        ulonglong2 s = load_slot(t.slots + i);
        if (s.x == kEmpty) {
            uint64_t old = atomicCAS((unsigned long long *)&t.slots[i].x, kEmpty, key);
            if (old == kEmpty) { *created += 1; s.x = key; }
            else s.x = old;
        }
        if (s.x == key)
            return atomicAdd((unsigned long long *)&t.slots[i].y, (unsigned long long)inc) + inc;
        i = (i + 1) & (t.cap - 1);
    }
}

// counts[key[u]] += inc[u] for the lanes' U live entries, as table_add_many, and before[u] = the
// count the key held just before its increment (0 for a key created here).  Never defers: the
// caller reserved room.  Returns the number of keys created.
template <int U>
__device__ __forceinline__ uint32_t table_add_fetch_many(const TableView &t, const uint64_t (&key)[U], const uint64_t (&inc)[U],
                                                         uint32_t live, uint64_t (&before)[U]) {
    uint64_t idx[U];
    ulonglong2 a[U], b[U];
    uint32_t created = 0;
#pragma unroll
    for (int u = 0; u < U; ++u) {
        before[u] = 0;
        if (((live >> u) & 1u) && key[u] == kEmpty) { before[u] = table_add_fetch(t, key[u], inc[u], &created) - inc[u]; live &= ~(1u << u); }
        idx[u] = t.home(key[u]);
        if ((live >> u) & 1u) load_pair(t.slots + idx[u], a[u], b[u]);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        if (!((live >> u) & 1u)) continue;
        if (a[u].x == key[u]) before[u] = atomicAdd((unsigned long long *)&t.slots[idx[u]].y, (unsigned long long)inc[u]);
        else if (b[u].x == key[u]) before[u] = atomicAdd((unsigned long long *)&t.slots[idx[u] + 1].y, (unsigned long long)inc[u]);
        else before[u] = table_add_fetch(t, key[u], inc[u], &created) - inc[u];
    }
    return created;
}

// slot index of key, or -1
__device__ __forceinline__ int64_t table_find(const TableView &t, uint64_t key) {
    uint64_t i = t.home(key);
    for (uint64_t probe = 0; probe < t.cap; ++probe) {
        ulonglong2 s = load_slot(t.slots + i);
        if (s.x == key) return (int64_t)i;
        if (s.x == kEmpty) return -1;
        i = (i + 1) & (t.cap - 1);
    }
    return -1;
}

__device__ __forceinline__ bool table_contains(const TableView &t, uint64_t key) {
    if (key == kEmpty) return t.ctrl->side_present != 0;
    return table_find(t, key) >= 0;
}

__device__ __forceinline__ uint64_t table_get(const TableView &t, uint64_t key) {
    if (key == kEmpty) return t.ctrl->side_present ? t.ctrl->side_count : 0;
    int64_t i = table_find(t, key);
    return i < 0 ? 0 : __ldcg(&t.slots[i].y);
}

// U lookups per thread with all home-bucket loads in flight together (one dependent random
// sector each is what bounds get / set comparison; a thread that waits for one at a time
// leaves the memory system idle).  cnt[j] = count or 0; returns the found mask.
template <int U>
__device__ __forceinline__ uint32_t table_get_many(const TableView &t, const uint64_t (&key)[U], uint32_t live,
                                                   uint64_t (&cnt)[U]) {
    ulonglong2 s0[U], s1[U];
#pragma unroll
    for (int j = 0; j < U; ++j) {
        cnt[j] = 0;
        // dead and out-of-band keys load bucket 0: harmless, keeps the loads unconditional
        const uint64_t h = ((live >> j) & 1) && key[j] != kEmpty ? t.home(key[j]) : 0;
        load_pair(t.slots + h, s0[j], s1[j]);
    }
    uint32_t found = 0;
#pragma unroll
    for (int j = 0; j < U; ++j) {
        if (!((live >> j) & 1)) continue;
        const uint64_t k = key[j];
        if (k == kEmpty) {
            if (t.ctrl->side_present) { cnt[j] = t.ctrl->side_count; found |= 1u << j; }
        } else if (s0[j].x == k) { cnt[j] = s0[j].y; found |= 1u << j; }
        else if (s0[j].x == kEmpty) {}
        else if (s1[j].x == k) { cnt[j] = s1[j].y; found |= 1u << j; }
        else if (s1[j].x == kEmpty) {}
        else {  // displaced past its home bucket: walk on
            uint64_t i = (t.home(k) + 2) & (t.cap - 1);
            for (uint64_t probe = 2; probe < t.cap; ++probe) {
                const ulonglong2 s = load_slot(t.slots + i);
                if (s.x == k) { cnt[j] = s.y; found |= 1u << j; break; }
                if (s.x == kEmpty) break;
                i = (i + 1) & (t.cap - 1);
            }
        }
    }
    return found;
}

}  // namespace oxg
