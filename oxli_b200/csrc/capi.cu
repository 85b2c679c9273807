// capi.cu -- host side of the C ABI declared in include/oxli_b200.h.
//
// One DeviceCtx per GPU (streams, staging buffers, scratch), one oxg_table per
// count table.  Everything is plain CUDA runtime: no torch, no Thrust/CUB.
#include <algorithm>
#include <atomic>
#include <cerrno>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstddef>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <system_error>
#include <thread>
#include <vector>

#include <fcntl.h>
#include <unistd.h>

#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>

#include "../../include/oxli_b200.h"
#include "aggregate.cuh"
#include "consume.cuh"
#include "dump.cuh"
#include "scatter.cuh"
#include "klist.h"
#include "lookup.cuh"
#include "shard.cuh"
#include "sortexport.cuh"
#include "tableops.cuh"
#include "owned.h"

using namespace oxg;

namespace {

// Shards of one process wait for each other inside kernels on different streams; streams that
// share a hardware work queue would serialise a wait in front of the kernel it waits for.  The
// driver reads this when the context is created, so it is set when the library is loaded
// (never overriding the user's choice).
const int g_connections_set = setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);

thread_local std::string g_err;
std::atomic<uint64_t> g_launches{0};

oxg_status fail(oxg_status st, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return st;
}

#define CU(expr)                                                                             \
    do {                                                                                     \
        cudaError_t e__ = (expr);                                                            \
        if (e__ != cudaSuccess)                                                              \
            return fail(e__ == cudaErrorMemoryAllocation ? OXG_ERR_NOMEM : OXG_ERR_CUDA,     \
                        "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__,   \
                        __LINE__);                                                           \
    } while (0)
#define TRY(expr)                          \
    do {                                   \
        oxg_status s__ = (expr);           \
        if (s__ != OXG_OK) return s__;     \
    } while (0)
#define LAUNCHED() (g_launches.fetch_add(1, std::memory_order_relaxed))

// NVTX ranges around the stages of an ingest call (copy / scatter / aggregate / fused consume /
// replay / shard round), so that a timeline of the end-to-end step can be read; free without a
// profiler attached
struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

// host->device streaming granule: OXLI_B200_CHUNK_MB in 1..1024, anything else means the default
static const uint64_t kChunkBytes = [] {
    const char *e = getenv("OXLI_B200_CHUNK_MB");
    long mb = 64;
    if (e && *e) {
        char *end = nullptr;
        const long v = strtol(e, &end, 10);
        if (end && *end == '\0' && v >= 1 && v <= 1024) mb = v;
    }
    return (uint64_t)mb << 20;
}();
static const uint64_t kLaunchWindows = [] {  // windows per consume launch (bounds the overflow list); OXLI_B200_LAUNCH_MW for experiments
    const char *e = getenv("OXLI_B200_LAUNCH_MW");
    const long v = e && *e ? atol(e) : 64;
    return (uint64_t)(v >= 1 && v <= 1024 ? v : 64) << 20;
}();
constexpr uint64_t kSmallBatch = 1ull << 20;      // below this, reserve for the worst case up front
constexpr uint64_t kMinCap = 1024;
// Launches of at least this many windows go through the partitioned pipeline (pass A scatter,
// pass B aggregate + merge); smaller ones keep the fused kernel, whose fixed costs are lower.
// OXLI_B200_PIPELINE=fused|part overrides the choice (part still needs a specialised k).
constexpr uint64_t kPartMinWindows = 8ull << 20;
static int env_int(const char *name, int dflt) { const char *e = getenv(name); return e && *e ? atoi(e) : dflt; }
// 0 = by launch size, 1 = fused kernel only, 2 = partitioned whenever the k is specialised
static std::atomic<int> g_pipeline{[] {
    const char *e = getenv("OXLI_B200_PIPELINE");
    return e && !strcmp(e, "fused") ? 1 : e && !strcmp(e, "part") ? 2 : 0;
}()};
static std::atomic<uint32_t> g_parts_override{(uint32_t)env_int("OXLI_B200_PARTS", 0)};    // 0 = from the table size
// pass A launches whose fragments pass B takes together (more duplicates per key meet in one
// aggregation, one merge instead of several); 1 = pass B after every pass A
static std::atomic<uint32_t> g_accumulate{(uint32_t)std::max(1, std::min(16, env_int("OXLI_B200_ACCUMULATE", 8)))};
static std::atomic<uint32_t> g_groups_override{(uint32_t)env_int("OXLI_B200_GROUPS", 0)};  // 0 = default
constexpr int kStageBufs = 4;  // host batches: chunks in flight between the copy stream and the kernels

// A host batch as the staging ring reads it: read boundaries offsets[0..n_reads] (positions in
// `bases`; the batch's own positions count from offsets[0]) and whether `bases` is pinned.
struct HostBatch {
    const uint8_t *bases;
    const uint64_t *offsets;
    uint64_t n_reads;
    bool pinned;
};

// Ring of kStageBufs staging buffers through which host batches reach the device: chunk ci goes
// to buffer ci % kStageBufs.  A buffer holds the chunk's bases (through pinned memory when the
// source is pageable) and its batch-relative read boundaries; ev_ready[b] marks its copies
// landed, ev_free[b] (recorded by whoever launches the kernels) the kernels done reading it.
struct StageRing {
    DeviceArray<uint8_t> d_bases[kStageBufs];
    PinnedArray<uint8_t> h_bases[kStageBufs];
    DeviceArray<uint64_t> d_offs[kStageBufs];
    PinnedArray<uint64_t> h_offs[kStageBufs];
    uint64_t n_off[kStageBufs] = {};  // boundaries of the chunk staged in buffer b, sentinel included
    Event ev_ready[kStageBufs], ev_free[kStageBufs];
    Stream copy;  // the H2D copies (declared last: drained and gone before the buffers it reads)

    oxg_status init() {
        CU(copy.create(cudaStreamNonBlocking));
        for (int b = 0; b < kStageBufs; ++b) { CU(ev_ready[b].create(cudaEventDisableTiming)); CU(ev_free[b].create(cudaEventDisableTiming)); }
        return OXG_OK;
    }

    // Buffers 0..n_bufs-1 take chunks of `bytes`.  A device buffer is replaced once `kernels` has
    // drained, a pinned one (needed for pageable sources only) once the copy stream has.
    oxg_status reserve(int n_bufs, uint64_t bytes, bool src_pinned, cudaStream_t kernels) {
        for (int b = 0; b < n_bufs; ++b) {
            if (d_bases[b].cap() < bytes) { CU(cudaStreamSynchronize(kernels)); CU(d_bases[b].reserve(bytes)); }
            if (!src_pinned && h_bases[b].cap() < bytes) { CU(cudaStreamSynchronize(copy)); CU(h_bases[b].reserve(bytes)); }
        }
        return OXG_OK;
    }

    // room for n boundaries in buffer b; `kernels` (if any) is drained too before the old ones go
    oxg_status reserve_offs(int b, uint64_t n, cudaStream_t kernels) {
        if (d_offs[b].cap() >= n && h_offs[b].cap() >= n) return OXG_OK;
        CU(cudaStreamSynchronize(copy));
        if (kernels) CU(cudaStreamSynchronize(kernels));
        CU(d_offs[b].reserve(n, 1 << 16)); CU(h_offs[b].reserve(n, 1 << 16));
        return OXG_OK;
    }

    // Stage bytes [lo, hi) of batch h (batch-relative) as chunk ci of n_chunks: queue the copies
    // of the bases and of the read boundaries that can fall inside [lo, hi + 1] on the copy
    // stream.  The caller makes its kernels wait for ev_ready[b] and records ev_free[b] after them.
    oxg_status stage(const HostBatch &h, uint64_t ci, uint64_t n_chunks, uint64_t lo, uint64_t hi, cudaStream_t kernels) {
        const int b = (int)(ci % kStageBufs);
        const uint64_t base0 = h.offsets[0];
        // every chunk also validates its share of the offsets (all pairs are seen once per call),
        // so the O(n_reads) pass runs next to the copies instead of in front of the first one
        for (uint64_t r = h.n_reads * ci / n_chunks, e = h.n_reads * (ci + 1) / n_chunks; r < e; ++r)
            if (h.offsets[r + 1] < h.offsets[r]) return fail(OXG_ERR_INVALID, "offsets must be non-decreasing");
        const uint64_t *ob = std::lower_bound(h.offsets, h.offsets + h.n_reads + 1, base0 + lo + 1);
        const uint64_t n = (uint64_t)(std::upper_bound(h.offsets, h.offsets + h.n_reads + 1, base0 + hi + 1) - ob);
        if (ci >= (uint64_t)kStageBufs) {
            // the buffer's previous chunk: its copy out of the pinned staging has finished (host
            // side may be refilled) and its kernels have read the device side
            CU(cudaEventSynchronize(ev_ready[b]));
            CU(cudaStreamWaitEvent(copy, ev_free[b], 0));
        }
        TRY(reserve_offs(b, n + 1, kernels));
        for (uint64_t i = 0; i < n; ++i) h_offs[b].get()[i] = ob[i] - base0;
        h_offs[b].get()[n] = ~0ULL >> 1;  // sentinel keeps n_off >= 1
        n_off[b] = n + 1;
        const uint8_t *src = h.bases + base0 + lo;
        if (!h.pinned) { memcpy(h_bases[b].get(), src, hi - lo); src = h_bases[b].get(); }
        CU(cudaMemcpyAsync(d_bases[b].get(), src, hi - lo, cudaMemcpyHostToDevice, copy));
        CU(cudaMemcpyAsync(d_offs[b].get(), h_offs[b].get(), n_off[b] * 8, cudaMemcpyHostToDevice, copy));
        CU(cudaEventRecord(ev_ready[b], copy));
        return OXG_OK;
    }
};

// Deferred (key, increment) pairs of a table that ran into its load limit (drain_deferred): the
// list launches defer into, and the one a replay of it defers into.  Fixed lists are allocated
// once and never enlarged (a shard's: see oxg_table::pooled).
struct DeferLists {
    DeviceArray<ulonglong2> pairs, pairs2;
    bool fixed = false;
};

struct DeviceCtx {
    int dev = -1;
    int sms = 0;
    Stream stream;
    std::mutex mu;
    StageRing ring;  // host batches
    Event ev_t0, ev_t1, ev_mid, ev_user0, ev_user1;
    // scratch
    DeviceArray<uint64_t> d_tile_first;
    DeferLists defer;                 // tables of this context that are not shards
    DeviceArray<uint64_t> d_dense;    // kHistDense bins
    DeviceArray<uint64_t> d_big;
    DeviceArray<uint64_t> d_io;       // generic u64 in/out scratch (device)
    PinnedArray<uint64_t> h_io;       // pinned mirror
    DeviceArray<double> d_f64;        // 4 doubles
    DeviceArray<uint8_t> d_seq;       // hash_windows input
    // partitioned pipeline (pass A output): fragments, their fill counts, the spill list
    DeviceArray<uint64_t> d_frag;
    DeviceArray<uint32_t> d_frag_cnt;
    DeviceArray<uint64_t> d_spill;
    DeviceArray<unsigned long long> d_spill_n;
    // export: compacted pairs, the second pair of arrays of the radix sort, its histogram, pinned bounce buffers
    DeviceArray<uint64_t> d_exp_k[2], d_exp_v[2];
    DeviceArray<uint64_t> d_exp_counts;
    DeviceArray<uint64_t> d_sort_hist;
    PinnedArray<uint8_t> h_bounce[2];
    Event ev_bounce[2];
};

// never destroyed: their owners would release after the CUDA runtime may have gone at exit
std::mutex g_ctx_mu;
std::vector<DeviceCtx *> g_ctx;

oxg_status get_ctx(int dev, DeviceCtx **out) {
    std::lock_guard<std::mutex> lk(g_ctx_mu);
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return fail(OXG_ERR_CUDA, "no CUDA device available (oxli_b200 has no CPU fallback)");
    }
    if (dev < 0 || dev >= n) return fail(OXG_ERR_INVALID, "device %d out of range (have %d)", dev, n);
    if ((int)g_ctx.size() < n) g_ctx.resize(n);
    if (!g_ctx[dev]) {
        auto c = std::make_unique<DeviceCtx>();
        c->dev = dev;
        CU(cudaSetDevice(dev));
        cudaDeviceProp prop;
        CU(cudaGetDeviceProperties(&prop, dev));
        if (prop.major < 10)
            return fail(OXG_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only",
                        dev, prop.major, prop.minor);
        c->sms = prop.multiProcessorCount;
        CU(c->stream.create(cudaStreamNonBlocking));
        TRY(c->ring.init());
        for (Event *e : {&c->ev_t0, &c->ev_t1, &c->ev_mid, &c->ev_user0, &c->ev_user1}) CU(e->create(cudaEventDefault));
        CU(c->d_dense.reserve(kHistDense));
        CU(c->d_f64.reserve(4));
        g_ctx[dev] = c.release();
    }
    *out = g_ctx[dev];
    return OXG_OK;
}

constexpr uint64_t kScratchMin = 1024;  // entries of a scratch array at least

oxg_status ensure_io(DeviceCtx *c, uint64_t n) {
    CU(c->d_io.reserve(n, kScratchMin));
    CU(c->h_io.reserve(n, kScratchMin));
    return OXG_OK;
}

int grid_for(const DeviceCtx *c, uint64_t items, int threads, int per_sm) {
    uint64_t want = (items + threads - 1) / threads;
    return (int)std::max<uint64_t>(1, std::min<uint64_t>(want, (uint64_t)c->sms * per_sm));
}

// Capacity policy.  Displaced keys are what slows the probe loop down
// (profiles/r1_microbench_probe_slow_path.txt: 16 % home-bucket misses at load
// 0.6 cut a 62 G keys/s loop to 23-35 G keys/s; at load 0.15 it runs at 66), so
// a table that is small anyway is kept sparse: up to kSparseBytes the target
// load is <= 0.3, beyond that memory and L2 footprint win and it may fill to 0.7.
constexpr uint64_t kSparseBytes = 128ull << 20;
uint64_t capacity_for_keys(uint64_t keys);
bool over_loaded(uint64_t size, uint64_t cap) {
    if (cap * 16 < kSparseBytes) return size * 10 > cap * 3;
    return size * 10 > cap * 7;
}

uint64_t pow2_at_least(uint64_t x) {
    uint64_t c = kMinCap;
    while (c < x) c <<= 1;
    return c;
}

uint64_t capacity_for_keys(uint64_t keys) {
    uint64_t cap = pow2_at_least(keys + keys / 2 + 1);                  // <= 67 % load
    while (cap * 16 < kSparseBytes && keys * 10 > cap * 3) cap <<= 1;   // sparse while it is cheap
    return cap;
}

// the slots of a table grown for `keys` distinct keys: <= 50 % load, and sparse while small
uint64_t slots_for(uint64_t keys) { return std::max(capacity_for_keys(keys), pow2_at_least(keys * 2)); }

// Device memory free now.  A slow driver call, and at times a very slow one (10-150 ms measured
// with two ranks on one box; asked in every round of the last third of a C3 step, it made steps of
// 95 ms take 100-260 ms at random): ask it only when there is a question.
oxg_status free_device_bytes(size_t *free_b) {
    size_t total = 0;
    CU(cudaMemGetInfo(free_b, &total));
    return OXG_OK;
}

// *yes: a table grown for `keys` would be larger than `cap` slots and take less than half of the
// free device memory (asked only when it would be larger)
oxg_status larger_and_fits(uint64_t keys, uint64_t cap, bool *yes) {
    *yes = false;
    const uint64_t want = slots_for(keys);
    if (want <= cap) return OXG_OK;
    size_t free_b = 0;
    TRY(free_device_bytes(&free_b));
    *yes = want * 16 < free_b / 2;
    return OXG_OK;
}


}  // namespace

namespace {
struct PartPlan {
    uint32_t n_parts = 0, part_bits = 0;   // partitions of one rank's table
    int n_ranks = 1, self_rank = 0, owner_shift = 64;
    uint32_t grid_a = 0;                   // CTAs of pass A = fragments per destination
    uint32_t frag_cap = 0;                 // entries per fragment (multiple of four: 32-byte sectors)
    uint32_t batch_tiles = 1;              // warp tiles per warp that pass A sorts by destination at a time
    uint64_t spill_cap = 0;
    uint32_t groups = 1;
    uint32_t n_dest() const { return n_parts * (uint32_t)n_ranks; }
    uint64_t frag_entries() const { return (uint64_t)n_dest() * grid_a * frag_cap; }
};

}  // namespace

struct oxg_table {
    DeviceCtx *ctx = nullptr;
    uint32_t k = 0;
    DeviceArray<ulonglong2> slots;  // (its capacity is the table's)
    DeviceArray<Ctrl> d_ctrl;
    PinnedArray<Ctrl> h_ctrl;
    uint64_t size = 0;       // host mirror of ctrl->size as of the last sync
    bool hinted = false;     // the caller said how many distinct keys to expect
    uint64_t hint_keys = 0;  // ... and this many
    bool pooled = false;     // slot arrays come from the stream-ordered allocator (shards: no call of
                             // theirs may synchronise the device while a peer's flag wait is running)
    float last_ms_a = 0.f, last_ms_b = 0.f;  // partitioned pipeline: pass A / pass B share of last_ms
    // partitioned pipeline: pass A launches whose fragments are waiting for their pass B
    struct {
        bool active = false;
        PartPlan pl;
        uint32_t launches = 0;
        uint64_t windows = 0, planned = 0;
    } pend;
    uint64_t part_budget = 0;  // windows the running consume call still has to go (0 = unknown)
    uint32_t group_cap = 0;    // != 0: at most this many pass A launches per pass B in the running call
    // HyperLogLog sketch of the keys that came in through the partitioned pipeline (aggregate.cuh)
    DeviceArray<uint32_t> d_sketch;
    PinnedArray<uint32_t> h_sketch;
    uint64_t sketch_covers = 0;    // keys of the table the sketch has seen
    uint64_t est_keys = 0;         // the sketch's last word on how many keys the table is about to hold
    uint64_t last_made = 0;        // keys the previous group of launches created
    uint64_t last_new = 0;   // keys created by the previous consume launch (growth look-ahead)
    float last_ms = 0.f;
    uint64_t last_launches = 0;
};

namespace {

// the table as its kernels see it; `defer` (nullptr: none) takes what runs into the load limit
TableView view_of(const oxg_table *t, const DeferLists *defer = nullptr) {
    TableView v;
    v.slots = t->slots.get();
    v.cap = t->slots.cap();
    uint32_t lg = 0;
    while ((1ull << lg) < t->slots.cap()) ++lg;
    v.shift = 64 - lg;
    v.limit = t->slots.cap() - t->slots.cap() / 5;  // stop creating keys at 80 % load
    v.ctrl = t->d_ctrl.get();
    v.overflow = defer ? defer->pairs.get() : nullptr;
    v.overflow_cap = defer ? defer->pairs.cap() : 0;
    return v;
}

oxg_status pull_ctrl(oxg_table *t) {
    DeviceCtx *c = t->ctx;
    CU(cudaMemcpyAsync(t->h_ctrl.get(), t->d_ctrl.get(), sizeof(Ctrl), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    t->size = t->h_ctrl.get()->size;
    return OXG_OK;
}

// zero the ctrl fields [first, first+n) (in uint64 units)
oxg_status zero_ctrl_fields(oxg_table *t, size_t first_field, size_t n_fields) {
    CU(cudaMemsetAsync(reinterpret_cast<uint64_t *>(t->d_ctrl.get()) + first_field, 0, n_fields * 8, t->ctx->stream));
    return OXG_OK;
}
constexpr size_t kFieldCounted = offsetof(Ctrl, counted) / 8;
constexpr size_t kFieldTile = offsetof(Ctrl, tile_counter) / 8;
constexpr size_t kLaunchFields = (offsetof(Ctrl, scratch) - offsetof(Ctrl, counted)) / 8;
constexpr size_t kFieldScratch = offsetof(Ctrl, scratch) / 8;

// a fresh slot array of cap slots, stream-ordered for a pooled table
oxg_status alloc_slots(const oxg_table *t, uint64_t cap, DeviceArray<ulonglong2> *out) {
    DeviceCtx *c = t->ctx;
    if (t->pooled) *out = DeviceArray<ulonglong2>(c->stream);  // (pools were 2x slower for growing multi-GB plain tables)
    CU(out->reserve(cap));
    init_slots_kernel<<<grid_for(c, cap, kOpThreads, 16), kOpThreads, 0, c->stream>>>(out->get(), cap);
    LAUNCHED();
    CU(cudaGetLastError());
    return OXG_OK;
}

// grow so that `keys` distinct keys sit at <= 50 % load
oxg_status grow_to_fit(oxg_table *t, uint64_t keys) {
    const uint64_t want = slots_for(keys);
    if (want <= t->slots.cap()) return OXG_OK;
    DeviceCtx *c = t->ctx;
    DeviceArray<ulonglong2> old;
    TRY(alloc_slots(t, want, &old));
    std::swap(t->slots, old);
    if (t->size) {
        rehash_kernel<<<grid_for(c, old.cap(), kOpThreads, 16), kOpThreads, 0, c->stream>>>(old.get(), old.cap(), view_of(t));
        LAUNCHED();
        CU(cudaGetLastError());
    }
    CU(cudaStreamSynchronize(c->stream));
    return OXG_OK;
}

oxg_status reserve_keys(oxg_table *t, uint64_t extra) { return grow_to_fit(t, t->size + extra); }

// Rebuild the table into a fresh slot array of the same size (erase, cut).  rebuild(old) queues
// the kernel that moves what stays from the old array into view_of(t) and adds what it drops to
// ctrl->scratch[0], which the caller has zeroed; side_drops(count) says whether the out-of-band
// key goes too.  *removed (if given): the keys dropped, the out-of-band one included.
template <class Rebuild, class SideDrops>
oxg_status rebuild_slots(oxg_table *t, const Rebuild &rebuild, const SideDrops &side_drops, uint64_t *removed) {
    DeviceArray<ulonglong2> old;
    TRY(alloc_slots(t, t->slots.cap(), &old));
    std::swap(t->slots, old);
    rebuild(old.get());
    LAUNCHED();
    CU(cudaGetLastError());
    TRY(pull_ctrl(t));
    old.reset();
    Ctrl *h = t->h_ctrl.get();
    uint64_t n = h->scratch[0];
    h->size -= n;
    if (h->side_present && side_drops(h->side_count)) { h->side_present = 0; h->side_count = 0; ++n; }
    t->size = h->size;
    CU(cudaMemcpyAsync(t->d_ctrl.get(), h, offsetof(Ctrl, counted), cudaMemcpyHostToDevice, t->ctx->stream));
    CU(cudaStreamSynchronize(t->ctx->stream));
    if (removed) *removed = n;
    return OXG_OK;
}

// A launch ran into the load limit and deferred `ov` hash OCCURRENCES (not distinct keys: on
// high-coverage input every new key is deferred many times).  Grow geometrically -- room for
// at most as many new keys as the table already holds -- and replay; a replay that runs into
// the limit again defers into the second list, the two swap and the loop goes round once more.
// A replay that defers again although the table did not grow met a probe run longer than
// kMaxProbe: keys that share one home at every capacity, which no growth separates.  The last
// replay then gets room for every deferred key and no deferral list: without one there is no
// probe limit and no load limit, so it places them all.
oxg_status drain_deferred(oxg_table *t, DeferLists &d, uint64_t ov) {
    NvtxRange range("oxg:replay deferred");
    DeviceCtx *c = t->ctx;
    if (ov > d.pairs.cap()) return fail(OXG_ERR_CUDA, "internal: overflow list overrun");
    uint64_t prev = ~0ULL;
    while (ov) {
        const uint64_t room = std::min<uint64_t>(ov, std::max<uint64_t>(t->size, 1ull << 20));
        const uint64_t cap_before = t->slots.cap();
        TRY(grow_to_fit(t, t->size + room));
        const bool last = t->slots.cap() == cap_before && ov >= prev;
        if (last) TRY(grow_to_fit(t, t->size + ov));
        prev = ov;
        if (!last) {
            if (!d.fixed) CU(d.pairs2.reserve(ov, kScratchMin));
            else if (d.pairs2.cap() < ov) return fail(OXG_ERR_NOMEM, "deferral list too small for the replay");
        }
        TRY(zero_ctrl_fields(t, offsetof(Ctrl, overflow) / 8, 1));
        TableView v = view_of(t);
        if (!last) { v.overflow = d.pairs2.get(); v.overflow_cap = d.pairs2.cap(); }
        replay_pairs_kernel<<<grid_for(c, (ov + 3) / 4, kOpThreads, 8), kOpThreads, 0, c->stream>>>(v, d.pairs.get(), ov);
        LAUNCHED();
        CU(cudaGetLastError());
        TRY(pull_ctrl(t));
        ov = t->h_ctrl.get()->overflow;
        std::swap(d.pairs, d.pairs2);
    }
    return OXG_OK;
}

// The end of a counting launch, or of a group of `launches` of them, begun at ev_t0: read the
// control block, add the time, the launches and the k-mers counted to the tallies, and tell the
// time, the keys created and the hash occurrences deferred.
struct Counting { float ms = 0.f; uint64_t made = 0, ov = 0; };
oxg_status end_counting(oxg_table *t, uint64_t launches, uint64_t *counted, Counting *out) {
    DeviceCtx *c = t->ctx;
    CU(cudaEventRecord(c->ev_t1, c->stream));
    const uint64_t size_before = t->size;
    TRY(pull_ctrl(t));
    CU(cudaEventElapsedTime(&out->ms, c->ev_t0, c->ev_t1));
    t->last_ms += out->ms; t->last_launches += launches;
    if (counted) *counted += t->h_ctrl.get()->counted;
    out->made = t->size - size_before;
    out->ov = t->h_ctrl.get()->overflow;
    return OXG_OK;
}

// k values with a compile-time specialised consume kernel: klist.h.  Each lives in its own
// translation unit (consume_inst.cu) and is reached through its entry function.
#define OXG_DECLARE_ENTRY(KK) extern "C" const void *oxg_consume_entry_##KK(int mode);
OXG_FOR_EACH_K(OXG_DECLARE_ENTRY)
#undef OXG_DECLARE_ENTRY
const void *specialised_entry(uint32_t k, int mode) {
    switch (k) {
#define OXG_K_ENTRY(KK) case KK: return oxg_consume_entry_##KK(mode);
        OXG_FOR_EACH_K(OXG_K_ENTRY)
#undef OXG_K_ENTRY
    default:
        return nullptr;
    }
}
bool specialised_k(uint32_t k) { return specialised_entry(k, kModeCount) != nullptr; }
uint32_t tile_width(uint32_t k) { return specialised_k(k) ? kWarpTile : kTileW; }

// Static + dynamic shared memory of fn may pass 48 KB: opt in, once per function and device.
oxg_status max_dyn_smem(const void *fn, int dev, size_t bytes) {
    static std::mutex mu;
    static std::vector<std::pair<const void *, int>> done;
    std::lock_guard<std::mutex> lk(mu);
    const std::pair<const void *, int> key{fn, dev};
    if (std::find(done.begin(), done.end(), key) != done.end()) return OXG_OK;
    CU(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    done.push_back(key);
    return OXG_OK;
}

template <int MODE>
oxg_status launch_consume(oxg_table *t, const ConsumeParams &p) {
    DeviceCtx *c = t->ctx;
    const int k = (int)t->k;
    auto grid_of = [&](const void *fn, size_t smem) {
        int per_sm = 1;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kThreads, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
        const uint64_t tiles_per_cta = specialised_k(t->k) ? kThreads / 32 : 1;
        const uint64_t work = p.n_tiles;
        return (int)std::max<uint64_t>(1, std::min<uint64_t>((work + tiles_per_cta - 1) / tiles_per_cta, (uint64_t)c->sms * per_sm));
    };
    if (const void *fn = specialised_entry(t->k, MODE)) {
        const size_t dyn = consume_dyn_smem(MODE);
        if (dyn) TRY(max_dyn_smem(fn, c->dev, dyn));
        void *args[] = {const_cast<ConsumeParams *>(&p)};
        CU(cudaLaunchKernel(fn, dim3(grid_of(fn, dyn)), dim3(kThreads), args, dyn, c->stream));
    } else {
        const size_t smem = generic_smem_bytes(k);
        consume_generic_kernel<MODE><<<grid_of((const void *)consume_generic_kernel<MODE>, smem), kThreads, smem, c->stream>>>(p);
    }
    LAUNCHED();
    CU(cudaGetLastError());
    return OXG_OK;
}


// ---- partitioned pipeline: pass A (hash + scatter) and pass B (aggregate + merge) -----------

// pass A launches per pass B: eight when the reads are resident (pass B 8.0 instead of 9.2 ms per C2
// step), four when they stream in from the host (the last group's pass B is the tail of the call)
uint32_t group_launches(const oxg_table *t) {
    const uint32_t g = g_accumulate.load();
    return t->group_cap ? std::min(g, t->group_cap) : g;
}

// Which pipeline a counting launch of `span` windows takes.  Measured on one B200
// (profiles/r2_pipeline_choice.txt): the partitioned pipeline matches or beats the fused kernel
// everywhere but on small launches -- hot table (C2: 29.0 vs 31.0 ms per step), low-complexity
// input (every window the same k-mer: 30x before the fused kernel learnt to pre-reduce a warp's
// repeats, on a par since), and, with pass B updating the table directly from a few thousand work
// items, input where nearly every key is new (C3-shaped, 273 M keys in 8 GiB: 65 vs 99 ms) -- there
// the fused kernel's updates are random DRAM accesses issued between hashes, pass B's come
// partition by partition.  Small launches stay fused: two kernels and a pass over fragments do
// not pay below some millions of windows.
bool use_partitioned(const oxg_table *t, uint64_t span) {
    if (!specialised_entry(t->k, kModePart)) return false;
    const int choice = g_pipeline.load();
    if (choice == 1) return false;
    if (choice == 2) return true;
    if (t->pend.active) return true;  // a group in flight is completed the way it began
    return span >= kPartMinWindows;
}

// Partition count: 3072-6144 distinct keys per partition, so that the shared-memory table of
// pass B (16384 slots in buckets of four) holds a partition's keys at load 0.2-0.4 and duplicates
// meet there; at most max_parts (2048 over all ranks), because pass A keeps three words per
// destination in shared memory next to its batch of hashes.
uint32_t choose_parts(const oxg_table *t, uint32_t max_parts) {
    const uint32_t forced = g_parts_override.load();
    if (forced >= 2 && !(forced & (forced - 1))) return std::min(forced, std::max(max_parts, 2u));
    const uint64_t est = std::max(t->size + t->last_new, t->hint_keys);
    if (est == 0) return std::min<uint32_t>(1024, max_parts);  // nothing known: the middle of the range
    uint64_t parts = 64;
    while (parts < max_parts && parts * 6144 < est) parts <<= 1;
    return (uint32_t)std::min<uint64_t>(parts, max_parts);
}

// dynamic shared memory of scatter_kernel<k> (its per-warp tile buffers as ScatWarpBuf<K>)
size_t scatter_smem_rt(uint32_t k, uint32_t n_dest, uint32_t batch_tiles) {
    const uint32_t q = 8 * ((k + 7 + 7) / 8);
    const uint32_t bl = ((kWarpTile - 8 + q) + 15) / 16 * 16;
    return scatter_smem_bytes(n_dest, batch_tiles, (int)(2 * bl + 128));
}

// CTAs of pass A for a launch of n_tiles warp tiles: kScatCtasPerSm per SM, fewer when the launch
// has less than one tile per warp of the full grid (scatter_full_grid_tiles).  A launch of fewer
// tiles than one batch of the grid simply leaves the batch part empty.
uint64_t scatter_full_grid_tiles(const DeviceCtx *c) { return (uint64_t)c->sms * kScatCtasPerSm * kScatWarps; }
uint32_t scatter_grid(const DeviceCtx *c, uint64_t n_tiles) {
    return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((n_tiles + kScatWarps - 1) / kScatWarps, (uint64_t)c->sms * kScatCtasPerSm));
}

oxg_status plan_partitioned(oxg_table *t, uint64_t span, uint64_t n_tiles, int n_ranks, int self_rank, PartPlan *out) {
    DeviceCtx *c = t->ctx;
    PartPlan pl;
    // destinations are (rank, partition), at most 2048: pass A keeps its largest batch at every k up to there
    pl.n_parts = choose_parts(t, std::max(2u, 2048u / (uint32_t)n_ranks));
    while ((1u << pl.part_bits) < pl.n_parts) ++pl.part_bits;
    pl.n_ranks = n_ranks; pl.self_rank = self_rank;
    int lg = 0;
    while ((1 << lg) < n_ranks) ++lg;
    pl.owner_shift = 64 - lg;
    // the batch of pass A: as large as the shared memory of kScatCtasPerSm CTAs per SM allows
    pl.batch_tiles = kScatMaxBatchTiles;
    while (pl.batch_tiles > 1 && scatter_smem_rt(t->k, pl.n_dest(), pl.batch_tiles) * kScatCtasPerSm > 220u * 1024) --pl.batch_tiles;
    if (scatter_smem_rt(t->k, pl.n_dest(), pl.batch_tiles) * kScatCtasPerSm > 220u * 1024) return fail(OXG_ERR_INVALID, "internal: too many scatter destinations");
    pl.grid_a = scatter_grid(c, n_tiles);
    // pass B reads the fill counts of a partition's fragments into shared memory, at most kAggMaxFrags
    if (pl.grid_a * (uint64_t)kMaxSources > kAggMaxFrags) return fail(OXG_ERR_INVALID, "internal: more pass A CTAs than pass B can take");
    // a fragment holds its fair share of the launch's windows plus half again plus four standard
    // deviations; what does not fit (skew) goes to the spill list, which can take the whole launch
    // (rounded up to whole 32-byte sectors, so that every fragment starts on one)
    const uint64_t fair = span / ((uint64_t)pl.n_dest() * pl.grid_a) + 1;
    uint64_t sq = 1;
    while (sq * sq < fair) ++sq;
    pl.frag_cap = (uint32_t)((fair + fair / 2 + 4 * sq + 3) & ~(uint64_t)3);
    pl.spill_cap = span;
    // work items of pass B = partitions x groups: enough of them (four per SM) that the CTAs finish
    // together -- 256 partitions of a shard on 148 SMs would otherwise be two uneven waves
    const uint32_t forced_groups = g_groups_override.load();
    pl.groups = forced_groups ? forced_groups : std::max<uint32_t>(1, std::min<uint32_t>(8, (4u * (uint32_t)c->sms + pl.n_parts - 1) / pl.n_parts));
    if (pl.frag_entries() >> 32) return fail(OXG_ERR_INVALID, "internal: fragment buffer too large for one launch");
    *out = pl;
    return OXG_OK;
}

// scatter_kernel needs more than 48 KB of dynamic shared memory
oxg_status scatter_attr(DeviceCtx *c, uint32_t k) { return max_dyn_smem(specialised_entry(k, kModePart), c->dev, 227 * 1024); }

oxg_status ensure_part_buffers(DeviceCtx *c, const PartPlan &pl) {
    CU(c->d_frag.reserve(pl.frag_entries(), kScratchMin));
    CU(c->d_frag_cnt.reserve((uint64_t)pl.n_dest() * pl.grid_a, kScratchMin));
    CU(c->d_spill.reserve(pl.spill_cap, kScratchMin));
    CU(c->d_spill_n.reserve(1));
    return OXG_OK;
}

// pass A: p is a filled-in ConsumeParams (table.ctrl is where `counted` goes)
oxg_status launch_part_a(oxg_table *t, ConsumeParams p, const PartPlan &pl, uint64_t *d_frag, uint32_t *d_frag_cnt,
                         uint64_t *d_spill, unsigned long long *d_spill_n, cudaStream_t stream, bool append = false) {
    DeviceCtx *c = t->ctx;
    const void *fn = specialised_entry(t->k, kModePart);
    TRY(scatter_attr(c, t->k));
    const size_t dyn = scatter_smem_rt(t->k, pl.n_dest(), pl.batch_tiles);
    p.frag = d_frag; p.frag_cnt = d_frag_cnt; p.frag_cap = pl.frag_cap;
    p.n_parts = pl.n_parts; p.part_shift = 64 - pl.part_bits; p.n_dest = pl.n_dest(); p.batch_tiles = pl.batch_tiles;
    p.n_ranks = pl.n_ranks; p.self_rank = pl.self_rank; p.owner_shift = pl.owner_shift;
    p.spill = d_spill; p.spill_cap = pl.spill_cap; p.spill_n = d_spill_n;
    p.frag_append = append ? 1u : 0u;
    if (p.n_tiles >> 31) return fail(OXG_ERR_INVALID, "internal: too many tiles for one pass A launch");
    if (!append) CU(cudaMemsetAsync(d_spill_n, 0, 8, stream));
    void *args[] = {&p};
    CU(cudaLaunchKernel(fn, dim3(pl.grid_a), dim3(kScatThreads), args, dyn, stream));
    LAUNCHED();
    CU(cudaGetLastError());
    return OXG_OK;
}

// The aggregation kernel in two variants, one CTA per SM each.  With the shared-memory cache:
// kAggThreadsDefault threads.  Without it, the kernel is bound by the latency of its table loads
// and wants every thread it can get (C3-shaped input, pass B per step: 512 / 768 / 1024 threads =
// 46.2 / 35.3 / 32.4 ms).
constexpr int kAggThreadsDirect = 1024;
const void *const kAggCached = (const void *)aggregate_kernel<kAggThreadsDefault, true>;
const void *const kAggDirect = (const void *)aggregate_kernel<kAggThreadsDirect, false>;

// The shared-memory table of pass B pays when keys repeat inside what it is given -- at least two
// occurrences per key the table holds, is hinted to hold or (sketch) is about to hold -- and a
// partition's keys fit it: 16 Ki slots took 4.9 K keys per partition at 9.2 ms per C2 step and
// 9.8 K at 19.6.  Nothing known at all (no hint, no sketch yet): on.
uint32_t use_cache_for(const oxg_table *t, const PartPlan &pl, uint64_t windows) {
    const uint64_t keys = std::max(std::max(t->size, t->hint_keys), t->est_keys);
    return keys == 0 || (windows >= 2 * keys && keys <= 8192ull * pl.n_parts) ? 1u : 0u;
}

// Work items per partition.  With the cache on, as few as keep the SMs level (the plan's: every
// item empties and merges a cache).  With it off an item is just a share of the partition's
// hashes: some thousands of items of 40 thousand hashes or more measured best (C3-shaped input,
// 8 GiB table, pass B over 512 Mi hashes at a time: 1024 partitions x 1 / 3 / 12 / 25 / 50 / 148
// items = 60.5 / 40.2 / 39.0 / 41.7 / 48.5 / 74.0 ms per step; 256 x 37 / 148 = 37.9 / 43.9; a shard's
// 1024 partitions over 64 Mi hashes at a time: x 3 / 8 / 16 = 86.7 / 94.5 / 120.5 ms per step).
uint32_t aggregate_groups(const PartPlan &pl, uint32_t use_cache, uint64_t hashes) {
    if (use_cache || g_groups_override.load()) return pl.groups;
    const uint64_t items = std::max<uint64_t>(1, hashes / 40960);
    return (uint32_t)std::max<uint64_t>(pl.groups, std::min<uint64_t>(64, (items + pl.n_parts - 1) / pl.n_parts));
}

// what pass B (and the sketch) of plan pl's rank reads: n_src sources of pass A output -- one,
// this device's own, without sharding -- into table view v
AggParams agg_params(const TableView &v, const PartPlan &pl, const AggSource *src, int n_src) {
    AggParams a{};
    a.table = v;
    for (int s = 0; s < n_src; ++s) a.src[s] = src[s];
    a.n_src = n_src;
    a.n_parts = pl.n_parts; a.dest0 = (uint32_t)pl.self_rank * pl.n_parts; a.n_ctas = pl.grid_a;
    a.frag_cap = pl.frag_cap; a.part_bits = pl.part_bits; a.spill_cap = pl.spill_cap;
    a.owner_shift = pl.owner_shift; a.self_rank = pl.self_rank; a.n_ranks = pl.n_ranks;
    return a;
}

// pass B over `windows` hashes of n_src sources.  Grid: one CTA per SM and item at most (the
// cached kernel fills an SM's shared memory; the direct one is held to one CTA per SM by its
// registers).
oxg_status launch_part_b(oxg_table *t, const TableView &v, const PartPlan &pl, const AggSource *src, int n_src,
                         uint64_t windows, cudaStream_t stream) {
    DeviceCtx *c = t->ctx;
    AggParams a = agg_params(v, pl, src, n_src);
    a.work_counter = (unsigned long long *)&t->d_ctrl.get()->absorb_counter;
    a.use_cache = use_cache_for(t, pl, windows);
    a.groups = aggregate_groups(pl, a.use_cache, windows);
    const void *fn = a.use_cache ? kAggCached : kAggDirect;
    const int threads = a.use_cache ? kAggThreadsDefault : kAggThreadsDirect;
    const size_t smem = aggregate_smem_bytes(a.use_cache != 0);
    if (a.use_cache) TRY(max_dyn_smem(fn, c->dev, smem));
    int per_sm = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, threads, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
    const uint64_t items = (uint64_t)a.n_parts * a.groups;
    const int grid = (int)std::max<uint64_t>(1, std::min<uint64_t>(items, (uint64_t)c->sms * per_sm));
    void *args[] = {&a};
    CU(cudaLaunchKernel(fn, dim3(grid), dim3(threads), args, smem, stream));
    LAUNCHED();
    CU(cudaGetLastError());
    return OXG_OK;
}

// the table's sketch, zeroed on stream st when it is new
oxg_status ensure_sketch(oxg_table *t, cudaStream_t st) {
    if (t->h_sketch.get()) return OXG_OK;  // (allocated last)
    CU(t->d_sketch.reserve(kSketchRegs));
    CU(cudaMemsetAsync(t->d_sketch.get(), 0, kSketchRegs * 4, st));
    CU(t->h_sketch.reserve(kSketchRegs));
    return OXG_OK;
}

// HyperLogLog estimate from 2^kSketchBits registers (Flajolet et al.; linear counting below 2.5 m)
double sketch_estimate(const uint32_t *regs) {
    const double m = (double)kSketchRegs;
    double sum = 0.0;
    uint32_t zeros = 0;
    for (uint32_t i = 0; i < kSketchRegs; ++i) { sum += std::ldexp(1.0, -(int)regs[i]); zeros += regs[i] == 0; }
    const double alpha = 0.7213 / (1.0 + 1.079 / m);
    double e = alpha * m * m / sum;
    if (e <= 2.5 * m && zeros) e = m * std::log(m / (double)zeros);
    return e;
}

// Before pass B: fold the group's hashes into the table's sketch and make room for what the
// table will hold afterwards -- unless the caller's hint still covers it.  `src` as for pass B.
oxg_status presize_for_group(oxg_table *t, const PartPlan &pl, const AggSource *src, int n_src, cudaStream_t stream,
                             uint64_t arrivals = 0, uint64_t rounds_left = 1) {
    DeviceCtx *c = t->ctx;
    TRY(ensure_sketch(t, stream));
    sketch_kernel<<<c->sms * 2, 512, 0, stream>>>(agg_params(TableView{}, pl, src, n_src), t->d_sketch.get());
    LAUNCHED();
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(t->h_sketch.get(), t->d_sketch.get(), kSketchRegs * 4, cudaMemcpyDeviceToHost, stream));
    CU(cudaStreamSynchronize(stream));
    const uint64_t unseen = t->size > t->sketch_covers ? t->size - t->sketch_covers : 0;  // keys that came in another way
    const double est = sketch_estimate(t->h_sketch.get());
    t->est_keys = (uint64_t)est + unseen;
    // sharded tables call this with a sketch of one round (shard_round), with more rounds to come:
    // where nearly everything that arrives is new (a quarter or more), room for half that rate over
    // the whole batch, in one step (the rate falls as coverage builds up); else for the rounds in
    // flight before the host monitor catches up
    double headroom = 1.0;
    if (rounds_left > 1) headroom = est * 4 >= (double)arrivals ? std::max(4.0, 0.5 * (double)rounds_left) : (double)std::min<uint64_t>(4, rounds_left);
    uint64_t expect = (uint64_t)(est * 1.04 * headroom) + unseen + 1024;  // 1.04: three standard errors
    if (headroom > 4.0) {  // a guess that size must not cost more than half of what is free
        size_t free_b = 0;
        TRY(free_device_bytes(&free_b));
        while (headroom > 4.0 && slots_for(expect) * 16 > free_b / 2) {
            headroom /= 2;
            expect = (uint64_t)(est * 1.04 * std::max(headroom, 4.0)) + unseen + 1024;
        }
    }
    if (expect * 10 > t->slots.cap() * 7) TRY(grow_to_fit(t, expect));
    return OXG_OK;
}

// pass B for the pass A launches accumulated so far, then the bookkeeping of a counting launch
oxg_status flush_pending(oxg_table *t, uint64_t *counted) {
    if (!t->pend.active) return OXG_OK;
    NvtxRange range("oxg:aggregate (pass B)");
    DeviceCtx *c = t->ctx;
    t->pend.active = false;
    CU(cudaEventRecord(c->ev_mid, c->stream));
    const AggSource own{c->d_frag.get(), c->d_frag_cnt.get(), c->d_spill.get(), c->d_spill_n.get()};
    // The sketch costs a pass over the group's hashes (0.8 ms per 209 M): taken when the table's
    // size is anybody's guess -- no hint (or the hint is used up), and either nothing is known yet
    // or the room left would not take twice what the previous group created.
    const bool hint_holds = t->hinted && t->size <= t->hint_keys;
    const bool roomy = t->size != 0 && (t->size + 2 * t->last_made) * 10 <= t->slots.cap() * 7;
    const bool sketched = !hint_holds && !roomy;
    if (sketched) TRY(presize_for_group(t, t->pend.pl, &own, 1, c->stream));
    TRY(launch_part_b(t, view_of(t, &c->defer), t->pend.pl, &own, 1, t->pend.windows, c->stream));
    Counting r;
    TRY(end_counting(t, t->pend.launches, counted, &r));
    float ms_a = 0.f;
    CU(cudaEventElapsedTime(&ms_a, c->ev_t0, c->ev_mid));
    t->last_ms_a += ms_a; t->last_ms_b += r.ms - ms_a;
    const uint64_t made = r.made;
    // forecast for the next group: what this one created, unless the caller's hint still covers the table
    t->last_new = r.ov ? made + r.ov : (t->hinted && t->size <= t->hint_keys) ? 0 : made;
    if (r.ov) TRY(drain_deferred(t, c->defer, r.ov));
    t->last_made = made;
    if (sketched) t->sketch_covers = t->size;
    if (!hint_holds) {
        // Where keys keep coming (a quarter of the windows or more brought a new key), the rest of
        // the call will bring them at no more than this rate: make the room now, in one step,
        // rather than by doubling under load.  0.6: the rate of a read set falls as coverage builds
        // up (C3-shaped input: 0.39 new keys per window in the first group, 0.22 over the whole set).
        if (made * 4 >= t->pend.windows && t->part_budget && t->size * 20 >= t->slots.cap() * 7) {  // (only a table that is filling up)
            const uint64_t more = (uint64_t)((double)made / (double)t->pend.windows * 0.6 * (double)t->part_budget);
            const uint64_t want = t->size + more;
            bool grow = false;
            TRY(larger_and_fits(want, t->slots.cap(), &grow));
            if (grow) TRY(grow_to_fit(t, want));
        }
    }
    return OXG_OK;
}

// Run one mode over window starts [w_lo, w_hi) of a device-resident span.
// `bases` holds global positions [g0, data_end); offsets are global positions.
// kModeCount: loops launches of <= kLaunchWindows windows, growing the table and
// replaying deferred hashes between launches.  *counted accumulates.
oxg_status run_span(oxg_table *t, int mode, const uint8_t *d_bases, uint64_t g0, uint64_t w_lo,
                    uint64_t w_hi, uint64_t data_end, const uint64_t *d_offsets, uint64_t n_off,
                    uint64_t *hashes_out, uint64_t *counted) {
    DeviceCtx *c = t->ctx;
    if (w_hi <= w_lo) return OXG_OK;
    if ((reinterpret_cast<uintptr_t>(d_bases) & 15) || (g0 & 15))
        return fail(OXG_ERR_INVALID, "device base buffer must be 16-byte aligned");
    uint64_t lo = w_lo;
    while (lo < w_hi) {
        const uint64_t tile_base = std::max<uint64_t>(g0, lo & ~(uint64_t)15);
        uint64_t hi = std::min<uint64_t>(w_hi, tile_base + kLaunchWindows);
        const uint32_t tw = tile_width(t->k);
        const uint64_t n_tiles = (hi - tile_base + tw - 1) / tw;
        CU(c->d_tile_first.reserve(n_tiles, kScratchMin));
        if (mode == kModeCount) {
            const uint64_t span = hi - lo;
            // a launch that will not join the group of pass A launches in flight (too small for the
            // partitioned pipeline) must not share its launch counters: complete the group first
            if (t->pend.active && !use_partitioned(t, span)) TRY(flush_pending(t, counted));
            if (span <= kSmallBatch) TRY(reserve_keys(t, span));
            else {
                // Look ahead instead of running into the load limit mid-launch: a table nobody
                // sized gets at least one slot per 8 windows of a full launch (128 MiB for 64 Mi
                // windows: enough for high-coverage data, cheap if it is not), and if the
                // previous launch created keys at a rate that would cross the limit, grow now.
                if (!t->hinted && t->slots.cap() < pow2_at_least(span / 8)) TRY(grow_to_fit(t, span / 16));
                const uint64_t expect = t->size + t->last_new + t->last_new / 4;
                if (expect * 10 > t->slots.cap() * 7) TRY(grow_to_fit(t, expect));
                else if (over_loaded(t->size, t->slots.cap())) TRY(grow_to_fit(t, t->size));
            }
            CU(c->defer.pairs.reserve(std::max<uint64_t>(span, t->pend.active ? t->pend.planned : 0), kScratchMin));
            // counted, overflow, absorbed, tile and absorb counters -- unless a group of pass A
            // launches is accumulating into them
            if (!t->pend.active) TRY(zero_ctrl_fields(t, kFieldCounted, kLaunchFields));
        } else {
            TRY(zero_ctrl_fields(t, kFieldTile, 1));
        }
        ConsumeParams p{};
        p.bases = d_bases; p.g0 = g0; p.w_lo = lo; p.w_hi = hi; p.data_end = data_end;
        p.tile_base = tile_base; p.n_tiles = n_tiles; p.offsets = d_offsets; p.n_off = n_off;
        p.tile_first = c->d_tile_first.get(); p.table = view_of(t, mode == kModeCount ? &c->defer : nullptr);
        p.hashes_out = hashes_out ? hashes_out + (lo - w_lo) : nullptr; p.ksize = t->k;
        tile_first_kernel<<<(unsigned)((n_tiles + 255) / 256), 256, 0, c->stream>>>(d_offsets, n_off, tile_base, n_tiles, tw, c->d_tile_first.get());
        LAUNCHED();
        CU(cudaGetLastError());
        const bool part = mode == kModeCount && use_partitioned(t, hi - lo);
        if (part) {
            NvtxRange range("oxg:scatter (pass A)");
            // pass A now; pass B once the group of launches is complete (flush_pending)
            const uint64_t span = hi - lo;
            if (t->pend.active && t->pend.windows + span > t->pend.planned) TRY(flush_pending(t, counted));
            if (!t->pend.active) {
                const uint64_t planned = std::min<uint64_t>(std::max<uint64_t>(t->part_budget, span), (uint64_t)group_launches(t) * kLaunchWindows);
                TRY(plan_partitioned(t, planned, planned / tw + 1, 1, 0, &t->pend.pl));
                TRY(ensure_part_buffers(c, t->pend.pl));
                t->pend.active = true; t->pend.launches = 0; t->pend.windows = 0; t->pend.planned = planned;
                CU(cudaEventRecord(c->ev_t0, c->stream));
            }
            TRY(launch_part_a(t, p, t->pend.pl, c->d_frag.get(), c->d_frag_cnt.get(), c->d_spill.get(), c->d_spill_n.get(), c->stream, t->pend.launches > 0));
            t->pend.launches += 1; t->pend.windows += span;
            t->part_budget = t->part_budget > span ? t->part_budget - span : 0;
            if (t->pend.launches >= group_launches(t) || t->pend.windows >= t->pend.planned) TRY(flush_pending(t, counted));
            lo = hi;
            continue;
        }
        NvtxRange range(mode == kModeCount ? "oxg:consume (fused)" : mode == kModeHash ? "oxg:hash windows" : "oxg:first-bad scan");
        CU(cudaEventRecord(c->ev_t0, c->stream));
        if (mode == kModeCount) TRY(launch_consume<kModeCount>(t, p));
        else if (mode == kModeHash) TRY(launch_consume<kModeHash>(t, p));
        else TRY(launch_consume<kModeFirstBad>(t, p));
        if (mode == kModeCount) {
            Counting r;
            TRY(end_counting(t, 1, counted, &r));
            // what the next launch of this stream will probably create: the rate of the last
            // quarter of this one (high-coverage input finds its keys early and then stops
            // creating them; the whole-launch count would quadruple the table for nothing),
            // or everything it wanted when it ran into the limit
            t->last_new = (hi - lo) <= kSmallBatch ? 0 : r.ov ? r.made + r.ov : 4 * t->h_ctrl.get()->late_new;
            if (r.ov) TRY(drain_deferred(t, c->defer, r.ov));  // table hit its load limit: grow, then replay the deferred hashes
        }
        lo = hi;
    }
    return OXG_OK;
}

// ---- error mode (src/lib.rs:586-600): count up to the first window holding a bad byte ---------

// Pre-scan: prime ctrl->first_bad, run kModeFirstBad over the batch's n_win windows through
// `span` (see consume_batch), and return the first bad window (~0: none).
template <class Span>
oxg_status first_bad_window(oxg_table *t, const Span &span, uint64_t n_win, uint64_t total, uint64_t *fb) {
    t->h_ctrl.get()->first_bad = ~0ULL;
    CU(cudaMemcpyAsync(&t->d_ctrl.get()->first_bad, &t->h_ctrl.get()->first_bad, 8, cudaMemcpyHostToDevice, t->ctx->stream));
    TRY(span(kModeFirstBad, 0, n_win, total, nullptr));
    TRY(pull_ctrl(t));
    *fb = t->h_ctrl.get()->first_bad;
    return OXG_OK;
}

// The read r holding window fb -- the last r with offsets[r] <= fb -- and where it starts.  A host
// batch (h_offsets given) counts positions from h_offsets[0]; a device-resident one from the
// start of its buffer, and its boundaries are read back from d_offsets.
oxg_status read_of(DeviceCtx *c, const uint64_t *h_offsets, const uint64_t *d_offsets, uint64_t n_reads, uint64_t fb,
                   uint64_t *r, uint64_t *r_start) {
    std::vector<uint64_t> tmp;
    uint64_t base0 = 0;
    if (h_offsets) {
        base0 = h_offsets[0];
    } else {
        tmp.resize(n_reads + 1);
        CU(cudaMemcpyAsync(tmp.data(), d_offsets, (n_reads + 1) * 8, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        h_offsets = tmp.data();
    }
    *r = (uint64_t)(std::upper_bound(h_offsets, h_offsets + n_reads + 1, base0 + fb) - h_offsets) - 1;
    *r_start = h_offsets[*r] - base0;
    return OXG_OK;
}

oxg_status bad_kmer(uint64_t r, uint64_t pos, int64_t *err_read, uint64_t *err_pos) {
    if (err_read) *err_read = (int64_t)r;
    if (err_pos) *err_pos = pos;
    return fail(OXG_ERR_BAD_KMER, "bad k-mer encountered at position %llu", (unsigned long long)pos);
}

// Consume a batch of n_reads reads, `total` bases, into one table.  span(mode, w_lo, w_hi,
// data_end, counted) runs one mode over window starts [w_lo, w_hi) of the batch: run_span over a
// device-resident batch, stream_span over a host one.  Offsets as for read_of.  group_cap: see
// oxg_table::group_cap.
template <class Span>
oxg_status consume_batch(oxg_table *t, const Span &span, const uint64_t *h_offsets, const uint64_t *d_offsets,
                         uint64_t n_reads, uint64_t total, int skip_bad, uint32_t group_cap,
                         uint64_t *total_counted, int64_t *err_read, uint64_t *err_pos) {
    const uint64_t k = t->k;
    if (total_counted) *total_counted = 0;
    if (err_read) *err_read = -1;
    if (err_pos) *err_pos = 0;
    t->last_ms = 0.f; t->last_ms_a = 0.f; t->last_ms_b = 0.f; t->last_launches = 0;
    const uint64_t n_win = total >= k ? total - k + 1 : 0;
    if (n_win == 0) return OXG_OK;
    t->part_budget = n_win;
    t->group_cap = group_cap;
    uint64_t counted = 0, fb = ~0ULL;
    oxg_status ret = OXG_OK;
    if (!skip_bad) TRY(first_bad_window(t, span, n_win, total, &fb));
    if (fb == ~0ULL) {
        TRY(span(kModeCount, 0, n_win, total, &counted));
    } else {
        uint64_t r = 0, r_start = 0, in_read = 0;
        TRY(read_of(t->ctx, h_offsets, d_offsets, n_reads, fb, &r, &r_start));
        // everything before that read, then the clean prefix of the read itself
        TRY(span(kModeCount, 0, r_start >= k ? r_start - k + 1 : 0, r_start, &counted));
        TRY(flush_pending(t, &counted));  // the position reported below counts the windows of the bad read only
        TRY(span(kModeCount, r_start, fb, fb + k - 1, &in_read));
        TRY(flush_pending(t, &in_read));
        counted += in_read;
        ret = bad_kmer(r, in_read, err_read, err_pos);
    }
    if (ret == OXG_OK) TRY(flush_pending(t, &counted));
    t->part_budget = 0;
    t->group_cap = 0;
    if (total_counted) *total_counted = counted;
    return ret;
}

}  // namespace

// ------------------------------------------------------------------ C ABI ---

extern "C" {

const char *oxg_last_error(void) { return g_err.c_str(); }
const char *oxg_version(void) { return "0.3.0"; }  // tracks the reference's Cargo.toml version
int oxg_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
uint64_t oxg_launch_count(void) { return g_launches.load(); }
uint64_t oxg_live_allocations(void) { return g_owned_live.load(); }
uint64_t oxg_fail_allocation_after(uint64_t n) { return g_owned_fail_in.exchange(n); }

oxg_status oxg_table_create(int device, uint32_t ksize, uint64_t capacity_hint, oxg_table **out) {
    if (!out) return fail(OXG_ERR_INVALID, "out is null");
    *out = nullptr;
    if (ksize < 1 || ksize > 255) return fail(OXG_ERR_INVALID, "ksize must be in 1..255 (got %u)", ksize);
    DeviceCtx *c;
    TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->dev));
    auto t = std::make_unique<oxg_table>();
    t->ctx = c; t->k = ksize;
    t->hinted = capacity_hint != 0;
    t->hint_keys = capacity_hint;
    CU(t->d_ctrl.reserve(1));
    CU(cudaMemsetAsync(t->d_ctrl.get(), 0, sizeof(Ctrl), c->stream));
    CU(t->h_ctrl.reserve(1));
    memset(t->h_ctrl.get(), 0, sizeof(Ctrl));
    TRY(alloc_slots(t.get(), capacity_for_keys(capacity_hint), &t->slots));
    CU(cudaStreamSynchronize(c->stream));
    *out = t.release();
    return OXG_OK;
}

oxg_status oxg_table_destroy(oxg_table *t) {
    if (!t) return OXG_OK;
    std::lock_guard<std::mutex> lk(t->ctx->mu);
    cudaSetDevice(t->ctx->dev);
    cudaStreamSynchronize(t->ctx->stream);
    delete t;
    return OXG_OK;
}

#define ENTER(t)                                               \
    if (!(t)) return fail(OXG_ERR_INVALID, "table is null");   \
    DeviceCtx *c = (t)->ctx;                                   \
    std::lock_guard<std::mutex> lk(c->mu);                     \
    CU(cudaSetDevice(c->dev))

oxg_status oxg_table_clear(oxg_table *t) {
    ENTER(t);
    init_slots_kernel<<<grid_for(c, t->slots.cap(), kOpThreads, 16), kOpThreads, 0, c->stream>>>(t->slots.get(), t->slots.cap());
    LAUNCHED();
    CU(cudaGetLastError());
    CU(cudaMemsetAsync(t->d_ctrl.get(), 0, sizeof(Ctrl), c->stream));
    if (t->d_sketch.get()) CU(cudaMemsetAsync(t->d_sketch.get(), 0, kSketchRegs * 4, c->stream));
    t->sketch_covers = 0;
    t->est_keys = 0;
    t->last_made = 0;
    t->size = 0;
    t->last_new = 0;
    return OXG_OK;
}

oxg_status oxg_table_reserve(oxg_table *t, uint64_t n_keys) {
    ENTER(t);
    return grow_to_fit(t, std::max(n_keys, t->size));
}

oxg_status oxg_table_ksize(const oxg_table *t, uint32_t *ksize) {
    if (!t || !ksize) return fail(OXG_ERR_INVALID, "null argument");
    *ksize = t->k;
    return OXG_OK;
}

oxg_status oxg_table_capacity(const oxg_table *t, uint64_t *slots) {
    if (!t || !slots) return fail(OXG_ERR_INVALID, "null argument");
    *slots = t->slots.cap();
    return OXG_OK;
}

oxg_status oxg_sync(oxg_table *t) {
    ENTER(t);
    CU(cudaStreamSynchronize(c->stream));
    CU(cudaStreamSynchronize(c->ring.copy));
    return OXG_OK;
}

oxg_status oxg_timer_start(oxg_table *t) {
    ENTER(t);
    CU(cudaEventRecord(c->ev_user0, c->stream));
    return OXG_OK;
}

oxg_status oxg_timer_stop(oxg_table *t, float *ms) {
    ENTER(t);
    if (!ms) return fail(OXG_ERR_INVALID, "null argument");
    CU(cudaEventRecord(c->ev_user1, c->stream));
    CU(cudaEventSynchronize(c->ev_user1));
    CU(cudaEventElapsedTime(ms, c->ev_user0, c->ev_user1));
    return OXG_OK;
}

oxg_status oxg_last_consume_kernel_ms(oxg_table *t, float *ms, uint64_t *launches) {
    if (!t) return fail(OXG_ERR_INVALID, "table is null");
    if (ms) *ms = t->last_ms;
    if (launches) *launches = t->last_launches;
    return OXG_OK;
}

oxg_status oxg_set_pipeline(int choice, uint32_t n_parts, uint32_t groups) {
    if (choice < 0 || choice > 2) return fail(OXG_ERR_INVALID, "pipeline choice must be 0 (by size), 1 (fused) or 2 (partitioned)");
    if (n_parts && (n_parts < 2 || n_parts > 8192 || (n_parts & (n_parts - 1))))
        return fail(OXG_ERR_INVALID, "n_parts must be 0 or a power of two in 2..8192");
    g_pipeline.store(choice);
    g_parts_override.store(n_parts);
    g_groups_override.store(groups);
    return OXG_OK;
}

oxg_status oxg_last_consume_pass_ms(oxg_table *t, float *ms_scatter, float *ms_aggregate) {
    if (!t) return fail(OXG_ERR_INVALID, "table is null");
    if (ms_scatter) *ms_scatter = t->last_ms_a;
    if (ms_aggregate) *ms_aggregate = t->last_ms_b;
    return OXG_OK;
}

// ---- hashing ---------------------------------------------------------------

oxg_status oxg_hash_windows(oxg_table *t, const uint8_t *seq, uint64_t len, uint64_t *hashes_out) {
    ENTER(t);
    const uint64_t k = t->k;
    if (len < k) return OXG_OK;
    if (!seq || !hashes_out) return fail(OXG_ERR_INVALID, "null argument");
    const uint64_t n_win = len - k + 1;
    // piecewise so the device-side output stays bounded; scratch lives in the device context
    // (hash_kmer / count / get call this once per k-mer)
    const uint64_t piece = 4ull << 20;
    CU(c->d_seq.reserve(std::min(len, piece + k - 1) + 32, kScratchMin));
    TRY(ensure_io(c, std::min(n_win, piece) + 2));
    uint64_t *d_off = c->d_io.get() + std::min(n_win, piece);
    c->h_io.get()[0] = 0; c->h_io.get()[1] = len;
    CU(cudaMemcpyAsync(d_off, c->h_io.get(), 16, cudaMemcpyHostToDevice, c->stream));
    for (uint64_t lo = 0; lo < n_win; lo += piece) {
        const uint64_t hi = std::min(n_win, lo + piece);
        const uint64_t bytes = hi - lo + k - 1;
        CU(cudaMemcpyAsync(c->d_seq.get(), seq + lo, bytes, cudaMemcpyHostToDevice, c->stream));
        TRY(run_span(t, kModeHash, c->d_seq.get(), lo, lo, hi, lo + bytes, d_off, 2, c->d_io.get(), nullptr));
        CU(cudaMemcpyAsync(hashes_out + lo, c->d_io.get(), (hi - lo) * 8, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
    }
    return OXG_OK;
}

// ---- consume ---------------------------------------------------------------

oxg_status oxg_consume_batch_device(oxg_table *t, const uint8_t *d_bases, const uint64_t *d_offsets,
                                    uint64_t n_reads, uint64_t total_bases, int skip_bad,
                                    uint64_t *total_counted, int64_t *err_read, uint64_t *err_pos) {
    ENTER(t);
    if (total_counted) *total_counted = 0;
    if (n_reads == 0 || total_bases == 0) { if (err_read) *err_read = -1; if (err_pos) *err_pos = 0; return OXG_OK; }
    if (!d_bases || !d_offsets) return fail(OXG_ERR_INVALID, "null argument");
    auto span = [&](int mode, uint64_t w_lo, uint64_t w_hi, uint64_t data_end, uint64_t *counted) {
        return run_span(t, mode, d_bases, 0, w_lo, w_hi, data_end, d_offsets, n_reads + 1, nullptr, counted);
    };
    return consume_batch(t, span, nullptr, d_offsets, n_reads, total_bases, skip_bad, 0, total_counted, err_read, err_pos);
}

oxg_status oxg_hash_batch_device(oxg_table *t, const uint8_t *d_bases, const uint64_t *d_offsets,
                                 uint64_t n_reads, uint64_t total_bases, uint64_t *d_hashes_out) {
    ENTER(t);
    if (!d_bases || !d_offsets || !d_hashes_out) return fail(OXG_ERR_INVALID, "null argument");
    const uint64_t k = t->k;
    if (total_bases < k) return OXG_OK;
    TRY(run_span(t, kModeHash, d_bases, 0, 0, total_bases - k + 1, total_bases, d_offsets, n_reads + 1, d_hashes_out, nullptr));
    CU(cudaStreamSynchronize(c->stream));
    return OXG_OK;
}

// Host batch: stream [w_lo, w_hi) through the context's staging ring.  A producer thread slices
// the read boundaries, stages pageable sources into pinned memory and queues the H2D copies back
// to back on the copy stream, up to kStageBufs chunks ahead of the kernels; the calling thread
// launches each chunk's kernels as its copy lands (run_span blocks until they are done, which is
// also what frees the chunk's buffer).  With only one chunk in flight ahead the copy engine idled
// between chunks and the step was 19 ms longer than its kernels.
static oxg_status stream_span(oxg_table *t, int mode, const HostBatch &h, uint64_t w_lo, uint64_t w_hi,
                              uint64_t data_end, uint64_t *counted) {
    DeviceCtx *c = t->ctx;
    StageRing &ring = c->ring;
    const uint64_t k = t->k;
    if (w_hi <= w_lo) return OXG_OK;
    const uint64_t first = w_lo & ~(uint64_t)(kTileW - 1);
    const uint64_t n_chunks = (w_hi - first + kChunkBytes - 1) / kChunkBytes;
    // staging sized to the batch (pinning full chunks costs a third of a second; a caller
    // that hands over a few thousand reads should not pay it), full chunks once one is needed
    const uint64_t stage_bytes = std::min(pow2_at_least(std::max<uint64_t>(data_end - first, 1 << 20)), kChunkBytes) + 256 + 16;
    TRY(ring.reserve((int)std::min<uint64_t>(n_chunks, kStageBufs), stage_bytes, h.pinned, c->stream));
    auto chunk_lo = [&](uint64_t ci) { return first + ci * kChunkBytes; };
    auto chunk_hi = [&](uint64_t ci) { return std::min(data_end, chunk_lo(ci) + kChunkBytes + k - 1); };
    // the previous use of buffer b (chunk ci - kStageBufs) is over: its kernels were waited for
    // (a partitioned launch is only queued when run_span returns)
    auto issue_copy = [&](uint64_t ci) -> oxg_status {
        NvtxRange range("oxg:stage + H2D copy");
        return ring.stage(h, ci, n_chunks, chunk_lo(ci), chunk_hi(ci), nullptr);
    };
    auto run_chunk = [&](uint64_t ci) -> oxg_status {
        const int b = (int)(ci % kStageBufs);
        const uint64_t lo = chunk_lo(ci);
        CU(cudaStreamWaitEvent(c->stream, ring.ev_ready[b], 0));
        TRY(run_span(t, mode, ring.d_bases[b].get(), lo, std::max(lo, w_lo), std::min(w_hi, lo + kChunkBytes), chunk_hi(ci),
                     ring.d_offs[b].get(), ring.n_off[b], nullptr, counted));
        CU(cudaEventRecord(ring.ev_free[b], c->stream));
        return OXG_OK;
    };
    if (n_chunks == 1) {
        TRY(issue_copy(0));
        TRY(run_chunk(0));
        if (mode != kModeCount) TRY(pull_ctrl(t));  // see below: the buffer is free again when this returns
        return OXG_OK;
    }
    std::mutex mu;
    std::condition_variable cv;
    uint64_t issued = 0, done = 0;  // chunks whose copies are queued / whose kernels have finished
    bool stop = false;
    oxg_status producer_status = OXG_OK;
    std::string producer_err;  // g_err is thread-local: carry the producer's message across
    auto produce = [&] {
        cudaSetDevice(c->dev);
        for (uint64_t ci = 0; ci < n_chunks; ++ci) {
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return stop || ci < done + kStageBufs; });
                if (stop) return;
            }
            const oxg_status st = issue_copy(ci);
            std::lock_guard<std::mutex> lk(mu);
            if (st != OXG_OK) { producer_status = st; producer_err = g_err; issued = n_chunks; cv.notify_all(); return; }
            issued = ci + 1;
            cv.notify_all();
        }
    };
    std::thread producer;
    try {
        producer = std::thread(produce);
    } catch (const std::system_error &) {
        // no helper thread to be had: stage and run the chunks in turn
        for (uint64_t ci = 0; ci < n_chunks; ++ci) {
            TRY(issue_copy(ci));
            TRY(run_chunk(ci));
            if (mode != kModeCount) {
                TRY(pull_ctrl(t));
                if (mode == kModeFirstBad && t->h_ctrl.get()->first_bad != ~0ULL) break;
            }
        }
        return OXG_OK;
    }
    oxg_status st = OXG_OK;
    for (uint64_t ci = 0; ci < n_chunks && st == OXG_OK; ++ci) {
        {
            std::unique_lock<std::mutex> lk(mu);
            cv.wait(lk, [&] { return issued > ci; });
            if (producer_status != OXG_OK) { st = fail(producer_status, "%s", producer_err.c_str()); break; }
        }
        st = run_chunk(ci);
        bool found = false;
        if (st == OXG_OK && mode != kModeCount) {
            // only counting launches are waited for inside run_span; the buffer must not be
            // refilled before this chunk's kernel has read it.  A pre-scan that has found its
            // bad window needs no later chunk.
            st = pull_ctrl(t);
            found = st == OXG_OK && mode == kModeFirstBad && t->h_ctrl.get()->first_bad != ~0ULL;
        }
        std::lock_guard<std::mutex> lk(mu);
        done = ci + 1;
        cv.notify_all();
        if (found) break;
    }
    {
        std::lock_guard<std::mutex> lk(mu);
        stop = true;
        cv.notify_all();
    }
    producer.join();
    // a call that stopped early (error, or pre-scan hit) may have copies queued that nobody will
    // wait for: drain them before the staging buffers are used again
    if (st != OXG_OK || mode != kModeCount) cudaStreamSynchronize(ring.copy);
    return st;
}

oxg_status oxg_consume_batch(oxg_table *t, const uint8_t *bases, const uint64_t *offsets,
                             uint64_t n_reads, int skip_bad, uint64_t *total_counted,
                             int64_t *err_read, uint64_t *err_pos) {
    ENTER(t);
    if (total_counted) *total_counted = 0;
    if (err_read) *err_read = -1;
    if (err_pos) *err_pos = 0;
    if (n_reads == 0) return OXG_OK;
    if (!bases || !offsets) return fail(OXG_ERR_INVALID, "null argument");
    // (monotonicity of the offsets is checked chunk by chunk while they are staged: StageRing::stage)
    if (offsets[n_reads] < offsets[0]) return fail(OXG_ERR_INVALID, "offsets must be non-decreasing");
    cudaPointerAttributes attr{};
    const bool pinned = cudaPointerGetAttributes(&attr, bases) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    const HostBatch h{bases, offsets, n_reads, pinned};
    auto span = [&](int mode, uint64_t w_lo, uint64_t w_hi, uint64_t data_end, uint64_t *counted) {
        return stream_span(t, mode, h, w_lo, w_hi, data_end, counted);
    };
    return consume_batch(t, span, offsets, nullptr, n_reads, offsets[n_reads] - offsets[0], skip_bad, 4, total_counted, err_read, err_pos);
}


// ---- by-hash operations ----------------------------------------------------

// counts a device-resident hash list in launches of <= kLaunchWindows entries; large
// lists go in optimistically (load-limit deferral + growth + replay) like consume
static oxg_status count_list_device(oxg_table *t, const uint64_t *d_hashes, uint64_t n, int skip_zero, uint64_t *counted) {
    DeviceCtx *c = t->ctx;
    for (uint64_t lo = 0; lo < n; lo += kLaunchWindows) {
        const uint64_t m = std::min<uint64_t>(kLaunchWindows, n - lo);
        const bool optimistic = m > kSmallBatch;
        if (!optimistic) TRY(reserve_keys(t, m));
        else {
            if (over_loaded(t->size, t->slots.cap())) TRY(grow_to_fit(t, t->size));
            CU(c->defer.pairs.reserve(m, kScratchMin));
        }
        TRY(zero_ctrl_fields(t, kFieldCounted, kLaunchFields));
        CU(cudaEventRecord(c->ev_t0, c->stream));
        count_hashes_kernel<<<grid_for(c, (m + 7) / 8, kOpThreads, 8), kOpThreads, 0, c->stream>>>(view_of(t, optimistic ? &c->defer : nullptr), d_hashes + lo, m, nullptr, skip_zero);
        LAUNCHED();
        CU(cudaGetLastError());
        Counting r;
        TRY(end_counting(t, 1, counted, &r));
        if (r.ov) TRY(drain_deferred(t, c->defer, r.ov));
    }
    return OXG_OK;
}

oxg_status oxg_count_hashes_device(oxg_table *t, const uint64_t *d_hashes, uint64_t n, int skip_zero, uint64_t *n_counted) {
    ENTER(t);
    if (n_counted) *n_counted = 0;
    if (n == 0) return OXG_OK;
    if (!d_hashes) return fail(OXG_ERR_INVALID, "null argument");
    t->last_ms = 0.f; t->last_ms_a = 0.f; t->last_ms_b = 0.f; t->last_launches = 0;
    return count_list_device(t, d_hashes, n, skip_zero, n_counted);
}

oxg_status oxg_count_hashes(oxg_table *t, const uint64_t *hashes, uint64_t n, uint64_t *new_counts) {
    ENTER(t);
    if (n == 0) return OXG_OK;
    if (!hashes) return fail(OXG_ERR_INVALID, "null argument");
    TRY(reserve_keys(t, n));
    TRY(ensure_io(c, 2 * n));
    memcpy(c->h_io.get(), hashes, n * 8);
    CU(cudaMemcpyAsync(c->d_io.get(), c->h_io.get(), n * 8, cudaMemcpyHostToDevice, c->stream));
    count_hashes_kernel<<<grid_for(c, n, kOpThreads, 16), kOpThreads, 0, c->stream>>>(view_of(t), c->d_io.get(), n, new_counts ? c->d_io.get() + n : nullptr, 0);
    LAUNCHED();
    CU(cudaGetLastError());
    if (new_counts) CU(cudaMemcpyAsync(c->h_io.get() + n, c->d_io.get() + n, n * 8, cudaMemcpyDeviceToHost, c->stream));
    TRY(pull_ctrl(t));
    if (new_counts) memcpy(new_counts, c->h_io.get() + n, n * 8);
    return OXG_OK;
}

oxg_status oxg_add_pairs(oxg_table *t, const uint64_t *keys, const uint64_t *vals, uint64_t n) {
    ENTER(t);
    if (n == 0) return OXG_OK;
    if (!keys || !vals) return fail(OXG_ERR_INVALID, "null argument");
    TRY(reserve_keys(t, n));
    TRY(ensure_io(c, 2 * n));
    memcpy(c->h_io.get(), keys, n * 8);
    memcpy(c->h_io.get() + n, vals, n * 8);
    CU(cudaMemcpyAsync(c->d_io.get(), c->h_io.get(), 2 * n * 8, cudaMemcpyHostToDevice, c->stream));
    add_pairs_kernel<<<grid_for(c, n, kOpThreads, 16), kOpThreads, 0, c->stream>>>(view_of(t), c->d_io.get(), c->d_io.get() + n, n);
    LAUNCHED();
    CU(cudaGetLastError());
    // the out-of-band key's side entry must exist even when its value is 0
    for (uint64_t i = 0; i < n; ++i)
        if (keys[i] == kEmpty) { const uint64_t one = 1; CU(cudaMemcpyAsync(&t->d_ctrl.get()->side_present, &one, 8, cudaMemcpyHostToDevice, c->stream)); break; }
    return pull_ctrl(t);
}

oxg_status oxg_get_hashes(oxg_table *t, const uint64_t *hashes, uint64_t n, uint64_t *counts_out) {
    ENTER(t);
    if (n == 0) return OXG_OK;
    if (!hashes || !counts_out) return fail(OXG_ERR_INVALID, "null argument");
    TRY(ensure_io(c, 2 * n));
    memcpy(c->h_io.get(), hashes, n * 8);
    CU(cudaMemcpyAsync(c->d_io.get(), c->h_io.get(), n * 8, cudaMemcpyHostToDevice, c->stream));
    get_hashes_kernel<<<grid_for(c, n, kOpThreads, 16), kOpThreads, 0, c->stream>>>(view_of(t), c->d_io.get(), n, c->d_io.get() + n);
    LAUNCHED();
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(c->h_io.get() + n, c->d_io.get() + n, n * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    memcpy(counts_out, c->h_io.get() + n, n * 8);
    return OXG_OK;
}

oxg_status oxg_set_hash(oxg_table *t, uint64_t hash, uint64_t value) {
    ENTER(t);
    TRY(reserve_keys(t, 1));
    set_hash_kernel<<<1, 32, 0, c->stream>>>(view_of(t), hash, value);
    LAUNCHED();
    CU(cudaGetLastError());
    return pull_ctrl(t);
}

oxg_status oxg_erase_hashes(oxg_table *t, const uint64_t *hashes, uint64_t n, uint64_t *n_removed) {
    ENTER(t);
    if (n_removed) *n_removed = 0;
    if (n == 0) return OXG_OK;
    if (!hashes) return fail(OXG_ERR_INVALID, "null argument");
    TRY(ensure_io(c, n));
    memcpy(c->h_io.get(), hashes, n * 8);
    CU(cudaMemcpyAsync(c->d_io.get(), c->h_io.get(), n * 8, cudaMemcpyHostToDevice, c->stream));
    if (n < 256) {
        // the reference's usage: one key per call (drop / drop_hash, src/lib.rs:197-224)
        erase_hashes_kernel<<<1, 32, 0, c->stream>>>(view_of(t), c->d_io.get(), n);
        LAUNCHED();
        CU(cudaGetLastError());
        TRY(pull_ctrl(t));
        if (n_removed) *n_removed = t->h_ctrl.get()->scratch[0];
        return OXG_OK;
    }
    // a list: mark in parallel, rebuild once
    TRY(pull_ctrl(t));
    DeviceArray<uint32_t> doomed;
    const uint64_t words = (t->slots.cap() + 31) / 32;
    CU(doomed.reserve(words));
    CU(cudaMemsetAsync(doomed.get(), 0, words * 4, c->stream));
    TRY(zero_ctrl_fields(t, kFieldScratch, 1));
    erase_mark_kernel<<<grid_for(c, n, kOpThreads, 16), kOpThreads, 0, c->stream>>>(view_of(t), c->d_io.get(), n, doomed.get());
    LAUNCHED();
    TRY(rebuild_slots(t, [&](const ulonglong2 *old) {
        erase_rebuild_kernel<<<grid_for(c, t->slots.cap(), kOpThreads, 16), kOpThreads, 0, c->stream>>>(old, t->slots.cap(), view_of(t), doomed.get());
    }, [&](uint64_t) { return std::find(hashes, hashes + n, kEmpty) != hashes + n; }, n_removed));
    return OXG_OK;
}

oxg_status oxg_cut(oxg_table *t, int mode, uint64_t thresh, uint64_t *n_removed) {
    ENTER(t);
    if (mode != 0 && mode != 1) return fail(OXG_ERR_INVALID, "mode must be 0 (mincut) or 1 (maxcut)");
    TRY(pull_ctrl(t));
    TRY(zero_ctrl_fields(t, kFieldScratch, 1));
    return rebuild_slots(t, [&](const ulonglong2 *old) {
        cut_kernel<<<grid_for(c, t->slots.cap(), kOpThreads, 16), kOpThreads, 0, c->stream>>>(old, t->slots.cap(), view_of(t), mode, thresh);
    }, [&](uint64_t v) { return mode == 0 ? v < thresh : v > thresh; }, n_removed);
}

// ---- scans -------------------------------------------------------------------

static oxg_status run_stats(oxg_table *t, bool histo, oxg_stats *st, uint64_t *n_big) {
    DeviceCtx *c = t->ctx;
    if (histo) {
        CU(cudaMemsetAsync(c->d_dense.get(), 0, kHistDense * 8, c->stream));
        if (!c->d_big.get()) CU(c->d_big.reserve(1 << 16));
    }
    for (int attempt = 0; attempt < 2; ++attempt) {
        Ctrl init{};
        init.scratch[2] = ~0ULL;
        memcpy(t->h_ctrl.get()->scratch, init.scratch, sizeof init.scratch);
        CU(cudaMemcpyAsync(t->d_ctrl.get()->scratch, t->h_ctrl.get()->scratch, sizeof init.scratch, cudaMemcpyHostToDevice, c->stream));
        stats_kernel<<<grid_for(c, t->slots.cap(), kOpThreads, 8), kOpThreads, 0, c->stream>>>(view_of(t), histo ? c->d_dense.get() : nullptr, c->d_big.get(), c->d_big.cap());
        LAUNCHED();
        CU(cudaGetLastError());
        TRY(pull_ctrl(t));
        if (!histo || t->h_ctrl.get()->scratch[4] <= c->d_big.cap()) break;
        // more huge counts than the list holds: enlarge and redo
        CU(c->d_big.reserve(t->h_ctrl.get()->scratch[4], kScratchMin));
        CU(cudaMemsetAsync(c->d_dense.get(), 0, kHistDense * 8, c->stream));
    }
    const Ctrl *h = t->h_ctrl.get();
    st->len = h->scratch[0]; st->sum = h->scratch[1];
    st->min = h->scratch[0] ? h->scratch[2] : ~0ULL; st->max = h->scratch[3];
    if (h->side_present) {
        st->len += 1; st->sum += h->side_count;
        st->min = std::min(st->min, h->side_count); st->max = std::max(st->max, h->side_count);
    }
    if (st->len == 0) { st->min = 0; st->max = 0; }
    if (n_big) *n_big = h->scratch[4];
    return OXG_OK;
}

oxg_status oxg_table_len(oxg_table *t, uint64_t *len) {
    ENTER(t);
    if (!len) return fail(OXG_ERR_INVALID, "null argument");
    TRY(pull_ctrl(t));
    *len = t->h_ctrl.get()->size + (t->h_ctrl.get()->side_present ? 1 : 0);
    return OXG_OK;
}

oxg_status oxg_table_stats(oxg_table *t, oxg_stats *out) {
    ENTER(t);
    if (!out) return fail(OXG_ERR_INVALID, "null argument");
    return run_stats(t, false, out, nullptr);
}

oxg_status oxg_histo(oxg_table *t, uint64_t *freq, uint64_t *n, uint64_t cap, uint64_t *n_out) {
    ENTER(t);
    if (!n_out) return fail(OXG_ERR_INVALID, "null argument");
    oxg_stats st;
    uint64_t n_big = 0;
    TRY(run_stats(t, true, &st, &n_big));
    std::vector<uint64_t> dense(kHistDense), big(n_big);
    CU(cudaMemcpyAsync(dense.data(), c->d_dense.get(), kHistDense * 8, cudaMemcpyDeviceToHost, c->stream));
    if (n_big) CU(cudaMemcpyAsync(big.data(), c->d_big.get(), n_big * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (t->h_ctrl.get()->side_present) {
        const uint64_t v = t->h_ctrl.get()->side_count;
        if (v < kHistDense) dense[v] += 1; else big.push_back(v);
    }
    std::sort(big.begin(), big.end());
    uint64_t w = 0, total = 0;
    auto emit = [&](uint64_t f, uint64_t cnt) {
        if (w < cap && freq && n) { freq[w] = f; n[w] = cnt; ++w; }
        ++total;
    };
    for (uint64_t f = 0; f < kHistDense; ++f) if (dense[f]) emit(f, dense[f]);
    for (size_t i = 0; i < big.size();) {
        size_t j = i;
        while (j < big.size() && big[j] == big[i]) ++j;
        emit(big[i], j - i);
        i = j;
    }
    *n_out = total;
    return OXG_OK;
}

oxg_status oxg_table_digest(oxg_table *t, int n_ranks, int rank, uint64_t out[5]) {
    ENTER(t);
    if (!out) return fail(OXG_ERR_INVALID, "null argument");
    if (n_ranks < 1 || (n_ranks & (n_ranks - 1)) || rank < 0 || rank >= n_ranks) return fail(OXG_ERR_INVALID, "bad rank / n_ranks");
    int lg = 0;
    while ((1 << lg) < n_ranks) ++lg;
    CU(cudaMemsetAsync(t->d_ctrl.get()->scratch, 0, 5 * 8, c->stream));
    digest_kernel<<<grid_for(c, t->slots.cap(), kOpThreads, 8), kOpThreads, 0, c->stream>>>(view_of(t), 64 - lg, (uint64_t)rank);
    LAUNCHED();
    CU(cudaGetLastError());
    TRY(pull_ctrl(t));
    const Ctrl *h = t->h_ctrl.get();
    for (int i = 0; i < 5; ++i) out[i] = h->scratch[i];
    if (h->side_present) {  // the out-of-band key 2^64-1 (owner: the last rank)
        out[0] += 1; out[1] += h->side_count; out[2] ^= kEmpty; out[3] += kEmpty * h->side_count;
        if (n_ranks > 1 && rank != n_ranks - 1) out[4] += 1;
    }
    return OXG_OK;
}

// ---- export --------------------------------------------------------------------

constexpr uint64_t kBounceBytes = 32ull << 20;

// Where a table's pairs go on the device: [0] the compaction (size + 1 pairs: the side entry joins
// them), [1] the radix sort's second pair of arrays (size + 1), chunk counts of the compaction
// (export_chunks + 1), the sort's histogram (256 per sort tile).  The plain table passes its device
// context's arrays, a shard its own (shards on one device share the context).
struct ExportArrays {
    uint64_t *k[2] = {}, *v[2] = {};
    uint64_t *chunk_counts = nullptr;
    uint64_t *sort_hist = nullptr;
};

static uint64_t export_chunks(const oxg_table *t) { return (t->slots.cap() + kExportChunk - 1) / kExportChunk; }
static uint64_t sort_tiles(uint64_t n) { return (n + kSortTile - 1) / kSortTile; }

// ordered compaction of the live slots into a.k[0] / a.v[0] (room for out_cap pairs) on stream st
// (slot order: stable between calls while the table is not modified, so dump() == list(iter),
// src/lib.rs:330-381,658)
static oxg_status export_device(const oxg_table *t, cudaStream_t st, const ExportArrays &a, uint64_t out_cap, uint64_t *n_live) {
    const uint64_t n_chunks = export_chunks(t);
    export_count_kernel<<<(unsigned)n_chunks, kOpThreads, 0, st>>>(t->slots.get(), t->slots.cap(), a.chunk_counts);
    LAUNCHED();
    export_scan_kernel<<<1, 1024, 0, st>>>(a.chunk_counts, n_chunks, a.chunk_counts + n_chunks);
    LAUNCHED();
    CU(cudaGetLastError());
    uint64_t live = 0;
    CU(cudaMemcpyAsync(&live, a.chunk_counts + n_chunks, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (live >= out_cap) return fail(OXG_ERR_INVALID, "internal: %llu live slots, room for %llu", (unsigned long long)live, (unsigned long long)out_cap);
    export_write_kernel<<<(unsigned)n_chunks, kOpThreads, 0, st>>>(t->slots.get(), t->slots.cap(), a.chunk_counts, a.k[0], a.v[0], live, nullptr);
    LAUNCHED();
    CU(cudaGetLastError());
    *n_live = live;
    return OXG_OK;
}

// stable LSD radix sort of the n pairs in a.k[0] / a.v[0] on stream st; *which = the pair of arrays
// holding the result
static oxg_status sort_pairs_device(cudaStream_t st, const ExportArrays &a, uint64_t n, int sort_mode, uint64_t max_count, int *which) {
    *which = 0;
    if (n < 2) return OXG_OK;
    const uint64_t n_tiles = sort_tiles(n);
    int cur = 0;
    auto pass = [&](int shift, int by_count) -> oxg_status {
        radix_hist_kernel<<<(unsigned)n_tiles, kSortThreads, 0, st>>>(a.k[cur], a.v[cur], n, shift, by_count, n_tiles, a.sort_hist);
        LAUNCHED();
        radix_scan_kernel<<<1, 1024, 0, st>>>(a.sort_hist, 256 * n_tiles);
        LAUNCHED();
        radix_scatter_kernel<<<(unsigned)n_tiles, kSortThreads, 0, st>>>(a.k[cur], a.v[cur], a.k[cur ^ 1], a.v[cur ^ 1],
                                                                         n, shift, by_count, n_tiles, a.sort_hist);
        LAUNCHED();
        CU(cudaGetLastError());
        cur ^= 1;
        return OXG_OK;
    };
    for (int shift = 0; shift < 64; shift += 8) TRY(pass(shift, 0));           // by hash
    if (sort_mode == 2)                                                        // then, stably, by count
        for (int shift = 0; shift < 64 && (max_count >> shift) != 0; shift += 8) TRY(pass(shift, 1));
    *which = cur;
    return OXG_OK;
}

// A table's n pairs (side entry included: side_count when `side`) in sort_mode order in a.k[*which] /
// a.v[*which], on stream st.  Returns with st drained.
static oxg_status export_pairs_device(const oxg_table *t, cudaStream_t st, const ExportArrays &a, uint64_t out_cap, bool side,
                                      uint64_t side_count, int sort_mode, uint64_t max_count, uint64_t *n_out, int *which) {
    uint64_t n = 0;
    TRY(export_device(t, st, a, out_cap, &n));
    if (side) {  // the out-of-band key 2^64-1 lives outside the slot array: it joins the pairs here
        const uint64_t kv[2] = {kEmpty, side_count};
        CU(cudaMemcpyAsync(a.k[0] + n, &kv[0], 8, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(a.v[0] + n, &kv[1], 8, cudaMemcpyHostToDevice, st));
        ++n;
    }
    *which = 0;
    if (sort_mode != 0) TRY(sort_pairs_device(st, a, n, sort_mode, max_count, which));
    CU(cudaStreamSynchronize(st));
    *n_out = n;
    return OXG_OK;
}

// two pinned buffers of `bytes` each and an event per buffer, through which device memory reaches the host
struct Bounce {
    uint8_t *buf[2];
    cudaEvent_t ev[2];
    uint64_t bytes;
};

// `bytes` of device memory at d_src, piece by piece through the bounce buffers on stream st:
// sink(at, p, len) receives bytes [at, at + len) while the next piece is on its way
static oxg_status stream_to_host(cudaStream_t st, const Bounce &b, const uint8_t *d_src, uint64_t bytes,
                                 const std::function<oxg_status(uint64_t, const uint8_t *, uint64_t)> &sink) {
    const uint64_t per = b.bytes;
    const uint64_t n_pieces = (bytes + per - 1) / per;
    for (uint64_t i = 0; i <= n_pieces; ++i) {
        if (i < n_pieces) {
            const uint64_t lo = i * per, cnt = std::min(per, bytes - lo);
            CU(cudaMemcpyAsync(b.buf[i & 1], d_src + lo, cnt, cudaMemcpyDeviceToHost, st));
            CU(cudaEventRecord(b.ev[i & 1], st));
        }
        if (i > 0) {  // piece i-1 has landed while piece i is on its way
            const uint64_t lo = (i - 1) * per, cnt = std::min(per, bytes - lo);
            CU(cudaEventSynchronize(b.ev[(i - 1) & 1]));
            TRY(sink(lo, b.buf[(i - 1) & 1], cnt));
        }
    }
    return OXG_OK;
}

// device array -> caller's host array through the bounce buffers (the caller's memory is usually
// pageable: a plain cudaMemcpy would stage it the same way, but one chunk at a time)
static oxg_status download(cudaStream_t st, const Bounce &b, uint64_t *dst, const uint64_t *d_src, uint64_t n) {
    if (!dst || n == 0) return OXG_OK;
    return stream_to_host(st, b, reinterpret_cast<const uint8_t *>(d_src), n * 8, [&](uint64_t at, const uint8_t *p, uint64_t len) {
        memcpy(reinterpret_cast<uint8_t *>(dst) + at, p, len);
        return OXG_OK;
    });
}

oxg_status oxg_export(oxg_table *t, uint64_t *keys, uint64_t *vals, uint64_t cap, int sort_mode, uint64_t *n_out) {
    ENTER(t);
    if (!n_out) return fail(OXG_ERR_INVALID, "null argument");
    if (sort_mode < 0 || sort_mode > 2) return fail(OXG_ERR_INVALID, "sort_mode must be 0, 1 or 2");
    TRY(pull_ctrl(t));
    const bool side = t->h_ctrl.get()->side_present != 0;
    const uint64_t side_count = t->h_ctrl.get()->side_count;
    const uint64_t live = t->h_ctrl.get()->size, total = live + (side ? 1 : 0);
    *n_out = total;
    if (cap == 0 || total == 0) return OXG_OK;
    uint64_t max_count = 0;
    if (sort_mode == 2) {
        oxg_stats st;
        TRY(run_stats(t, false, &st, nullptr));
        max_count = st.max;
    }
    // the context's export arrays, grown as needed
    CU(c->d_exp_counts.reserve(export_chunks(t) + 1, kScratchMin));
    for (int i = 0; i < (sort_mode != 0 && total >= 2 ? 2 : 1); ++i) { CU(c->d_exp_k[i].reserve(live + 1)); CU(c->d_exp_v[i].reserve(live + 1)); }
    if (sort_mode != 0 && total >= 2) CU(c->d_sort_hist.reserve(256 * sort_tiles(total), kScratchMin));
    for (int b = 0; b < 2; ++b) { CU(c->h_bounce[b].reserve(kBounceBytes)); if (!c->ev_bounce[b]) CU(c->ev_bounce[b].create(cudaEventDisableTiming)); }
    const ExportArrays a{{c->d_exp_k[0].get(), c->d_exp_k[1].get()}, {c->d_exp_v[0].get(), c->d_exp_v[1].get()}, c->d_exp_counts.get(), c->d_sort_hist.get()};
    uint64_t n = 0;
    int which = 0;
    TRY(export_pairs_device(t, c->stream, a, std::min(c->d_exp_k[0].cap(), c->d_exp_v[0].cap()), side, side_count, sort_mode, max_count, &n, &which));
    const Bounce b{{c->h_bounce[0].get(), c->h_bounce[1].get()}, {c->ev_bounce[0], c->ev_bounce[1]}, kBounceBytes};
    TRY(download(c->stream, b, keys, a.k[which], std::min(n, cap)));
    TRY(download(c->stream, b, vals, a.v[which], std::min(n, cap)));
    CU(cudaStreamSynchronize(c->stream));
    return OXG_OK;
}

// ---- set comparisons -------------------------------------------------------------

static oxg_status two_tables(oxg_table *a, oxg_table *b) {
    if (!a || !b) return fail(OXG_ERR_INVALID, "table is null");
    if (a->ctx != b->ctx) return fail(OXG_ERR_INVALID, "tables live on different devices");
    return OXG_OK;
}

static oxg_status setop_sizes_locked(oxg_table *a, oxg_table *b, uint64_t *inter, uint64_t *uni) {
    DeviceCtx *c = a->ctx;
    TRY(pull_ctrl(b));
    TRY(zero_ctrl_fields(a, kFieldScratch, 1));
    setop_count_kernel<<<grid_for(c, a->slots.cap(), kOpThreads, 16), kOpThreads, 0, c->stream>>>(view_of(a), view_of(b));
    LAUNCHED();
    CU(cudaGetLastError());
    TRY(pull_ctrl(a));
    uint64_t both = a->h_ctrl.get()->scratch[0];
    if (a->h_ctrl.get()->side_present && b->h_ctrl.get()->side_present) both += 1;
    const uint64_t na = a->h_ctrl.get()->size + (a->h_ctrl.get()->side_present ? 1 : 0);
    const uint64_t nb = b->h_ctrl.get()->size + (b->h_ctrl.get()->side_present ? 1 : 0);
    if (inter) *inter = both;
    if (uni) *uni = na + nb - both;
    return OXG_OK;
}

oxg_status oxg_setop_sizes(oxg_table *a, oxg_table *b, uint64_t *inter, uint64_t *uni) {
    TRY(two_tables(a, b));
    ENTER(a);
    return setop_sizes_locked(a, b, inter, uni);
}

oxg_status oxg_jaccard(oxg_table *a, oxg_table *b, double *out) {
    TRY(two_tables(a, b));
    ENTER(a);
    if (!out) return fail(OXG_ERR_INVALID, "null argument");
    uint64_t inter = 0, uni = 0;
    TRY(setop_sizes_locked(a, b, &inter, &uni));
    *out = uni == 0 ? 1.0 : (double)inter / (double)uni;  // src/lib.rs:716-721
    return OXG_OK;
}

// Where the keys of a set operation go on the device: the mask of a pass (one bit per slot of the
// larger table), its chunk counts (export_chunks of the larger table + 1), the keys.
struct SetopArrays {
    uint16_t *mask = nullptr;
    uint64_t *chunk_counts = nullptr;
    uint64_t *keys = nullptr;
};

static uint64_t setop_chunks(const oxg_table *a, const oxg_table *b) { return std::max(export_chunks(a), export_chunks(b)); }

// One compaction on stream st: the live slots of x -- all of them (y == nullptr, the export's count)
// or those whose membership in y equals want_in_y -- in slot order at keys[*n ..), *n advanced.
static oxg_status setop_pass(const oxg_table *x, const oxg_table *y, int want_in_y, cudaStream_t st, const SetopArrays &a,
                             uint64_t out_cap, uint64_t *n) {
    const uint64_t n_chunks = export_chunks(x);
    if (y) setop_mask_kernel<<<(unsigned)n_chunks, kOpThreads, 0, st>>>(view_of(x), view_of(y), want_in_y, a.mask, a.chunk_counts);
    else export_count_kernel<<<(unsigned)n_chunks, kOpThreads, 0, st>>>(x->slots.get(), x->slots.cap(), a.chunk_counts);
    LAUNCHED();
    export_scan_kernel<<<1, 1024, 0, st>>>(a.chunk_counts, n_chunks, a.chunk_counts + n_chunks);
    LAUNCHED();
    CU(cudaGetLastError());
    uint64_t got = 0;
    CU(cudaMemcpyAsync(&got, a.chunk_counts + n_chunks, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (*n + got > out_cap) return fail(OXG_ERR_INVALID, "internal: %llu set keys, room for %llu", (unsigned long long)(*n + got), (unsigned long long)out_cap);
    export_write_kernel<<<(unsigned)n_chunks, kOpThreads, 0, st>>>(x->slots.get(), x->slots.cap(), a.chunk_counts, a.keys + *n, nullptr,
                                                                   out_cap - *n, y ? a.mask : nullptr);
    LAUNCHED();
    CU(cudaGetLastError());
    *n += got;
    return OXG_OK;
}

// The slot keys of a op b (an oxg_setop) in a.keys, each pass's in slot order, on stream st: *n of
// them.  2^64-1 lives outside the slot arrays: see setop_side.
static oxg_status setop_keys_device(const oxg_table *a, const oxg_table *b, int op, cudaStream_t st, const SetopArrays &arr,
                                    uint64_t out_cap, uint64_t *n) {
    *n = 0;
    switch (op) {
    case OXG_UNION: TRY(setop_pass(a, nullptr, 0, st, arr, out_cap, n)); return setop_pass(b, a, 0, st, arr, out_cap, n);
    case OXG_INTERSECTION: return setop_pass(a, b, 1, st, arr, out_cap, n);
    case OXG_DIFFERENCE: return setop_pass(a, b, 0, st, arr, out_cap, n);
    default: TRY(setop_pass(a, b, 0, st, arr, out_cap, n)); return setop_pass(b, a, 0, st, arr, out_cap, n);
    }
}

// whether the out-of-band key 2^64-1 is in a op b, given whether each table holds it
static bool setop_side(int op, bool sa, bool sb) {
    switch (op) {
    case OXG_UNION: return sa || sb;
    case OXG_INTERSECTION: return sa && sb;
    case OXG_DIFFERENCE: return sa && !sb;
    default: return sa != sb;
    }
}

oxg_status oxg_setop_export(oxg_table *a, oxg_table *b, int op, uint64_t *keys_out, uint64_t cap, uint64_t *n_out) {
    TRY(two_tables(a, b));
    ENTER(a);
    if (!n_out) return fail(OXG_ERR_INVALID, "null argument");
    if (op < 0 || op > 3) return fail(OXG_ERR_INVALID, "unknown set operation %d", op);
    TRY(pull_ctrl(a));
    TRY(pull_ctrl(b));
    const uint64_t room = a->h_ctrl.get()->size + b->h_ctrl.get()->size;
    const uint64_t n_chunks = setop_chunks(a, b);
    DeviceArray<uint16_t> mask;
    DeviceArray<uint64_t> counts, out;
    CU(mask.reserve(n_chunks * kOpThreads));
    CU(counts.reserve(n_chunks + 1));
    CU(out.reserve(room, 1));
    for (int i = 0; i < 2; ++i) { CU(c->h_bounce[i].reserve(kBounceBytes)); if (!c->ev_bounce[i]) CU(c->ev_bounce[i].create(cudaEventDisableTiming)); }
    uint64_t n = 0;
    TRY(setop_keys_device(a, b, op, c->stream, SetopArrays{mask.get(), counts.get(), out.get()}, room, &n));
    const bool side = setop_side(op, a->h_ctrl.get()->side_present != 0, b->h_ctrl.get()->side_present != 0);
    *n_out = n + (side ? 1 : 0);
    const Bounce bb{{c->h_bounce[0].get(), c->h_bounce[1].get()}, {c->ev_bounce[0], c->ev_bounce[1]}, kBounceBytes};
    TRY(download(c->stream, bb, keys_out, out.get(), std::min(n, cap)));
    if (keys_out && side && n < cap) keys_out[n] = kEmpty;  // the out-of-band key comes last
    return OXG_OK;
}

// The raw terms of cosine(a, b) (src/lib.rs:727-765), side entries included: the dot product over
// A & B (wrapping u64), sum a^2 and sum b^2 as doubles, |A| and |B|.  Locks a's context.
struct CosineTerms {
    uint64_t dot = 0;
    double sq_a = 0.0, sq_b = 0.0;
    uint64_t n_a = 0, n_b = 0;
};

static oxg_status cosine_terms(oxg_table *a, oxg_table *b, CosineTerms *out) {
    ENTER(a);
    TRY(pull_ctrl(a));
    TRY(pull_ctrl(b));
    const Ctrl ha = *a->h_ctrl.get(), hb = *b->h_ctrl.get();
    CosineTerms t;
    t.n_a = ha.size + (ha.side_present ? 1 : 0);
    t.n_b = hb.size + (hb.side_present ? 1 : 0);
    double sq[2] = {0.0, 0.0};
    if (ha.size || hb.size) {
        CU(cudaMemsetAsync(c->d_f64.get(), 0, 4 * sizeof(double), c->stream));
        TRY(zero_ctrl_fields(a, kFieldScratch, 1));
        cosine_kernel<<<grid_for(c, a->slots.cap(), kOpThreads, 16), kOpThreads, 0, c->stream>>>(view_of(a), view_of(b), c->d_f64.get());
        LAUNCHED();
        TableView none = view_of(a);
        none.slots = nullptr;  // norm-only pass over b: adds nothing to any dot product
        cosine_kernel<<<grid_for(c, b->slots.cap(), kOpThreads, 16), kOpThreads, 0, c->stream>>>(view_of(b), none, c->d_f64.get() + 1);
        LAUNCHED();
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(sq, c->d_f64.get(), 16, cudaMemcpyDeviceToHost, c->stream));
        TRY(pull_ctrl(a));
        t.dot = a->h_ctrl.get()->scratch[0];
    }
    if (ha.side_present) {
        sq[0] += (double)ha.side_count * (double)ha.side_count;
        if (hb.side_present) t.dot += ha.side_count * hb.side_count;
    }
    if (hb.side_present) sq[1] += (double)hb.side_count * (double)hb.side_count;
    t.sq_a = sq[0];
    t.sq_b = sq[1];
    *out = t;
    return OXG_OK;
}

// cosine from its terms: 0.0 when either table is empty (src/lib.rs:729-731) or a norm is 0
static double cosine_of(const CosineTerms &t) {
    if (t.n_a == 0 || t.n_b == 0) return 0.0;
    const double ma = sqrt(t.sq_a), mb = sqrt(t.sq_b);
    return (ma == 0.0 || mb == 0.0) ? 0.0 : (double)t.dot / (ma * mb);
}

oxg_status oxg_cosine(oxg_table *a, oxg_table *b, double *out) {
    TRY(two_tables(a, b));
    if (!out) return fail(OXG_ERR_INVALID, "null argument");
    CosineTerms t;
    TRY(cosine_terms(a, b, &t));
    *out = cosine_of(t);
    return OXG_OK;
}

oxg_status oxg_merge(oxg_table *dst, oxg_table *src, uint64_t *counts_added, uint64_t *new_keys) {
    TRY(two_tables(dst, src));
    if (dst == src) return fail(OXG_ERR_INVALID, "cannot merge a table into itself");
    if (dst->k != src->k) return fail(OXG_ERR_WRONG_KSIZE, "KmerCountTables must have the same ksize");
    ENTER(dst);
    TRY(pull_ctrl(dst));
    TRY(pull_ctrl(src));
    TRY(reserve_keys(dst, src->h_ctrl.get()->size));
    TRY(zero_ctrl_fields(dst, kFieldScratch, 2));
    merge_kernel<<<grid_for(c, src->slots.cap(), kOpThreads, 16), kOpThreads, 0, c->stream>>>(view_of(dst), view_of(src));
    LAUNCHED();
    CU(cudaGetLastError());
    TRY(pull_ctrl(dst));
    uint64_t added = dst->h_ctrl.get()->scratch[0], fresh = dst->h_ctrl.get()->scratch[1];
    if (src->h_ctrl.get()->side_present) {
        Ctrl *h = dst->h_ctrl.get();
        if (!h->side_present || h->side_count == 0) ++fresh;
        h->side_present = 1;
        h->side_count += src->h_ctrl.get()->side_count;
        added += src->h_ctrl.get()->side_count;
        CU(cudaMemcpyAsync(&dst->d_ctrl.get()->side_present, &h->side_present, 16, cudaMemcpyHostToDevice, c->stream));
        CU(cudaStreamSynchronize(c->stream));
    }
    if (counts_added) *counts_added = added;
    if (new_keys) *new_keys = fresh;
    return OXG_OK;
}

// ---- synthetic reads, memory helpers ------------------------------------------------

oxg_status oxg_synth_reads_device(int device, uint8_t *d_bases, uint64_t n_reads, uint32_t read_len,
                                  uint64_t genome_len, uint64_t seed, uint64_t first_read,
                                  uint32_t sub_ppm, uint32_t n_ppm) {
    DeviceCtx *c;
    TRY(get_ctx(device, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->dev));
    if (!d_bases || read_len == 0 || genome_len < read_len) return fail(OXG_ERR_INVALID, "bad synth arguments");
    synth_reads_kernel<<<c->sms * 16, 256, 0, c->stream>>>(d_bases, n_reads, read_len, genome_len, seed, first_read, sub_ppm, n_ppm);
    LAUNCHED();
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream));
    return OXG_OK;
}

oxg_status oxg_pinned_alloc(uint64_t bytes, void **out) {
    if (!out) return fail(OXG_ERR_INVALID, "null argument");
    CU(cudaMallocHost(out, bytes ? bytes : 1));
    return OXG_OK;
}
oxg_status oxg_pinned_free(void *p) {
    if (p) CU(cudaFreeHost(p));
    return OXG_OK;
}
oxg_status oxg_device_alloc(int device, uint64_t bytes, void **d_out) {
    DeviceCtx *c;
    TRY(get_ctx(device, &c));
    CU(cudaSetDevice(c->dev));
    CU(cudaMalloc(d_out, bytes ? bytes : 16));
    return OXG_OK;
}
oxg_status oxg_device_free(int device, void *d_ptr) {
    DeviceCtx *c;
    TRY(get_ctx(device, &c));
    CU(cudaSetDevice(c->dev));
    if (d_ptr) CU(cudaFree(d_ptr));
    return OXG_OK;
}
oxg_status oxg_memcpy_h2d(int device, void *d_dst, const void *src, uint64_t bytes) {
    DeviceCtx *c;
    TRY(get_ctx(device, &c));
    CU(cudaSetDevice(c->dev));
    CU(cudaMemcpy(d_dst, src, bytes, cudaMemcpyHostToDevice));
    return OXG_OK;
}
oxg_status oxg_memcpy_d2h(int device, void *dst, const void *d_src, uint64_t bytes) {
    DeviceCtx *c;
    TRY(get_ctx(device, &c));
    CU(cudaSetDevice(c->dev));
    CU(cudaMemcpy(dst, d_src, bytes, cudaMemcpyDeviceToHost));
    return OXG_OK;
}

}  // extern "C"

#include "capi_shard.inc"
