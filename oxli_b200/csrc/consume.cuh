// consume.cuh -- the sliding-window kernels (K1 fused with K2).
//
// Replaces the hot loop of KmerCountTable::consume
// (/root/reference/src/lib.rs:576-600): SeqToHashes iterator step (validity,
// canonical choice, murmur) + `count_hash` per window.
//
// Work decomposition: the batch is one flat byte stream; every position is a
// candidate window start.  A CTA takes tiles of kTileW consecutive starts
// (+K-1 bytes of halo), stages them once in shared memory as
//   s_fw : upper-cased bytes                     (forward strand)
//   s_rc : complemented bytes, mirrored           (reverse strand, so the
//          reverse complement of any window is again a contiguous byte run)
//   s_bad: 1 bit per byte, set for non-ACGT / past-the-end bytes
//   s_end: 1 bit per byte, set on the last base of a read (CSR boundary)
// and each thread then owns kWPT consecutive windows: it pulls Q bytes per
// strand with 64-bit shared loads, derives each window's words with constant
// funnel shifts, decides fw-vs-rc on the byte-swapped leading word (full
// compare only on a tie), hashes, and probes the table.  A window is counted
// iff no bad bit lies in [p,p+K) and no end bit in [p,p+K-1).
#pragma once
#include <utility>

#include "hashing.cuh"
#include "table.cuh"

namespace oxg {

template <class F, int... I>
__device__ __forceinline__ void static_for_impl(F &&f, std::integer_sequence<int, I...>) {
    (f(std::integral_constant<int, I>{}), ...);
}
// f(integral_constant<int, 0>) ... f(integral_constant<int, N-1>), fully unrolled
template <int N, class F>
__device__ __forceinline__ void static_for(F &&f) {
    static_for_impl(f, std::make_integer_sequence<int, N>{});
}

#ifndef OXG_MIN_CTAS
#define OXG_MIN_CTAS 3  // resident CTAs per SM the specialised kernel is compiled for
#endif

constexpr int kTileW = 2048;  // window starts per tile
constexpr int kThreads = 256;
constexpr int kWPT = kTileW / kThreads;  // 8 consecutive windows per thread
static_assert(kWPT == 8, "bit-mask extraction assumes 8 windows per thread");
constexpr int kWarpTile = 32 * kWPT;  // window starts per warp tile in the specialised kernel
constexpr int kMaxRanks = 16;

enum Mode : int {
    kModeCount = 0,    // hash + count into the table
    kModeHash = 1,     // hash only, write one u64 per window (0 = bad window)
    kModeFirstBad = 2, // error-mode pre-scan: smallest in-read window holding a bad byte
    kModePart = 3      // hash + scatter into per-CTA fragments, one per table partition (pass A)
};

struct ConsumeParams {
    const uint8_t *bases;  // device; bases[0] is global byte position g0 (16-byte aligned)
    uint64_t g0;
    uint64_t w_lo, w_hi;   // window starts handled by this launch
    uint64_t data_end;     // one past the last byte that may be read / belongs to the batch
    uint64_t tile_base;    // global start of tile 0: multiple of 16, g0 <= tile_base <= w_lo
    uint64_t n_tiles;
    const uint64_t *offsets;  // CSR offsets (global positions), n_off entries, ascending
    uint64_t n_off;
    const uint64_t *tile_first;  // per tile: first index r with offsets[r] > tile start
    TableView table;
    uint64_t *hashes_out;  // kModeHash: hashes_out[w - w_lo]
    uint32_t ksize;        // generic kernel only
    // sharding (kModePart): owner(h) = h >> owner_shift
    int owner_shift;
    int self_rank;
    int n_ranks;
    // kModePart (pass A of the partitioned pipeline, see aggregate.cuh).  Destination of hash h:
    //   dest = owner(h) * n_parts + ((h * phi) >> part_shift)      owner(h) = h >> owner_shift, 0 with one rank
    // so a destination is (rank, contiguous segment of that rank's table).  Every CTA of
    // scatter_kernel (scatter.cuh) owns one fragment of frag_cap entries per destination:
    // frag[(dest * gridDim.x + blockIdx.x) * frag_cap ..]; a hash whose fragment is full goes to
    // the spill list.  frag_cnt[dest * gridDim.x + blockIdx.x] = entries written.
    uint64_t *frag;
    uint32_t *frag_cnt;
    uint32_t frag_cap;
    uint32_t n_parts;        // partitions per rank (power of two, >= 2)
    uint32_t part_shift;     // 64 - log2(n_parts)
    uint32_t n_dest;         // n_ranks * n_parts
    uint32_t batch_tiles;    // warp tiles per warp that scatter_kernel sorts by destination at a time (scatter.cuh)
    uint32_t frag_append;    // != 0: continue the fragments where frag_cnt says an earlier launch left them
    uint64_t *spill;
    uint64_t spill_cap;
    unsigned long long *spill_n;
};

static __global__ void tile_first_kernel(const uint64_t *__restrict__ offsets, uint64_t n_off,
                                  uint64_t tile_base, uint64_t n_tiles, uint32_t tile_w,
                                  uint64_t *__restrict__ tile_first) {
    uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    const uint64_t want = tile_base + t * tile_w + 1;  // first offsets[r] >= want
    uint64_t lo = 0, hi = n_off;
    while (lo < hi) {
        uint64_t mid = (lo + hi) >> 1;
        if (offsets[mid] < want) lo = mid + 1; else hi = mid;
    }
    tile_first[t] = lo;
}

__device__ __forceinline__ uint4 load_bases16(const ConsumeParams &p, uint64_t g) {
    if (g + 16 <= p.data_end) {
        return __ldcs(reinterpret_cast<const uint4 *>(p.bases + (g - p.g0)));
    }
    uint32_t w[4] = {0x4e4e4e4eu, 0x4e4e4e4eu, 0x4e4e4e4eu, 0x4e4e4e4eu};  // 'N'
    for (int b = 0; b < 16; ++b) {
        if (g + b < p.data_end) {
            uint32_t c = p.bases[g + b - p.g0];
            w[b >> 2] = (w[b >> 2] & ~(0xffu << (8 * (b & 3)))) | (c << (8 * (b & 3)));
        }
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// Stage 16 bytes: forward bytes at s_fw[16v..], mirrored complement at
// s_rc[BL-16-16v ..], 16 bad bits at s_bad[v].
template <int BL>
__device__ __forceinline__ void stage16_raw(const ConsumeParams &p, uint64_t w0, int v, uint4 raw, uint8_t *s_fw,
                                            uint8_t *s_rc, uint16_t *s_bad) {
    const uint64_t g = w0 + 16ull * v;
    uint32_t u[4] = {upper4(raw.x), upper4(raw.y), upper4(raw.z), upper4(raw.w)};
    uint32_t ok = acgt_mask4(u[0]) | (acgt_mask4(u[1]) << 4) | (acgt_mask4(u[2]) << 8) |
                  (acgt_mask4(u[3]) << 12);
    if (g + 16 > p.data_end) {  // bytes past the end are bad whatever they hold
        uint32_t keep = g >= p.data_end ? 0u : (0xffffu >> (16 - (uint32_t)(p.data_end - g)));
        ok &= keep;
    }
    *reinterpret_cast<uint4 *>(s_fw + 16 * v) = make_uint4(u[0], u[1], u[2], u[3]);
    *reinterpret_cast<uint4 *>(s_rc + BL - 16 - 16 * v) =
        make_uint4(bswap32(complement4(u[3])), bswap32(complement4(u[2])),
                   bswap32(complement4(u[1])), bswap32(complement4(u[0])));
    s_bad[v] = (uint16_t)(~ok);
}

template <int BL>
__device__ __forceinline__ void stage16(const ConsumeParams &p, uint64_t w0, int v, uint8_t *s_fw,
                                        uint8_t *s_rc, uint16_t *s_bad) {
    stage16_raw<BL>(p, w0, v, load_bases16(p, w0 + 16ull * v), s_fw, s_rc, s_bad);
}

// ---- cp.async (LDGSTS): global -> shared without passing through registers ----
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
#ifndef OXG_STREAM_EVICT_FIRST
#define OXG_STREAM_EVICT_FIRST 1
#endif
// The bases are read once; the table is what should stay in L2.  The streaming copies carry
// an evict-first policy so that 1.5 GB of reads per step do not push table sectors out.
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t pol;
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void cp_async16_zfill(void *smem, const void *gmem, uint32_t src_bytes, uint64_t pol) {
#if OXG_STREAM_EVICT_FIRST
    asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2, %3;" ::"r"(smem_u32(smem)), "l"(gmem), "r"(src_bytes), "l"(pol) : "memory");
#else
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem)), "l"(gmem), "r"(src_bytes) : "memory");
#endif
}
__device__ __forceinline__ void cp_async8(void *smem, const void *gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
// ---- bulk async copy (the TMA engine's 1-D form) + mbarrier: one lane moves a whole tile ----
#ifndef OXG_BULK_STAGE
#define OXG_BULK_STAGE 1
#endif
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *smem, const void *gmem, uint32_t bytes, uint64_t *bar, uint64_t pol) {
#if OXG_STREAM_EVICT_FIRST
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(smem_u32(smem)), "l"(gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(pol) : "memory");
#else
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem)), "l"(gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
#endif
}

__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Count up to kWPT hashes per thread (0 = nothing to count).
//
// Fast path: one 256-bit load fetches the key's home bucket (two 16-byte slots = one
// 32-byte sector); a hit in either slot is one RED.
//
// Slow path: keys displaced from their home bucket (16 % at load 0.6), new keys and
// the "table at its load limit" case go to a per-warp shared-memory queue that
// persists across tiles.  After every tile ONE probe round runs over the whole queue:
// each queued key looks at its next bucket; hits and inserts leave the queue, the rest
// stay with their position advanced.  A key on a long probe chain therefore costs one
// extra load per tile it rides along, instead of stalling its warp for the whole chain
// (an ablation of the first version showed the 15 % displaced keys costing 12 of 35 ms:
// every tile waited for its longest chain, ~6 dependent round trips).
constexpr int kTileBatch = 8;   // consecutive warp tiles handed out per atomic
constexpr int kQueueCap = 320;  // entries per warp; a tile adds at most kWPT*32 = 256

struct SlowQueue {
    uint64_t *key;   // [kQueueCap]
    uint8_t *skip;   // [kQueueCap] slots already ruled out, counted from the home slot
    uint32_t n;      // warp-uniform
};

__device__ __forceinline__ void count_fast8(const TableView &tv, const uint64_t (&h)[kWPT], SlowQueue &q,
                                            uint64_t &n_counted) {
    const int lane = threadIdx.x & 31;
    uint32_t pending = 0, restart = 0;
#pragma unroll
    for (int half = 0; half < kWPT / 4; ++half) {
        uint64_t idx[4];
        ulonglong2 a[4], b[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = half * 4 + u;
            idx[u] = tv.home(h[j]);
            if (h[j] != 0) load_pair(tv.slots + idx[u], a[u], b[u]);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = half * 4 + u;
            if (h[j] == 0) continue;  // bad window, or the reference's hash==0 skip (src/lib.rs:589)
            ++n_counted;
            // the out-of-band key equals the empty-slot marker: it must not "match" an empty
            // slot; the slow round hands it to table_add, which keeps it in the side entry
            if (h[j] == kEmpty) pending |= 1u << j;
            else if (a[u].x == h[j]) red_add64(&tv.slots[idx[u]].y, 1);
            else if (b[u].x == h[j]) red_add64(&tv.slots[idx[u] + 1].y, 1);
            else {
                pending |= 1u << j;
                // an empty slot in the home bucket means "maybe insert here": look at it again
                if (a[u].x == kEmpty || b[u].x == kEmpty) restart |= 1u << j;
            }
        }
    }
#pragma unroll
    for (int j = 0; j < kWPT; ++j) {
        const bool mine = (pending >> j) & 1u;
        const unsigned m = __ballot_sync(0xffffffffu, mine);
        if (mine) {
            const uint32_t at = q.n + __popc(m & ((1u << lane) - 1));
            q.key[at] = h[j];
            q.skip[at] = ((restart >> j) & 1u) ? 0 : 2;
        }
        q.n += __popc(m);
    }
}

// One probe round over the queue.  Survivors are compacted to the front (in place: the
// write cursor never passes the chunk being read, which is held in registers by then).
__device__ __forceinline__ void slow_round(const TableView &tv, SlowQueue &q, bool full, uint32_t &created) {
    const int lane = threadIdx.x & 31;
    __syncwarp();
    uint32_t out = 0;
    for (uint32_t base = 0; base < q.n; base += 32) {
        const uint32_t i = base + lane;
        const bool live = i < q.n;
        const uint64_t key = live ? q.key[i] : 0;
        const uint32_t skip = live ? q.skip[i] : 0;
        __syncwarp();
        bool again = false;
        if (live) {
            const uint64_t idx = (tv.home(key) + skip) & (tv.cap - 1);
            ulonglong2 a, b;
            load_pair(tv.slots + idx, a, b);
            if (key == kEmpty || skip >= 250) created += table_add(tv, key, 1, full);  // out-of-band key / absurd chain
            else if (a.x == key) red_add64(&tv.slots[idx].y, 1);
            else if (b.x == key) red_add64(&tv.slots[idx + 1].y, 1);
            else if (a.x == kEmpty || b.x == kEmpty) created += table_add(tv, key, 1, full);  // claim (or defer when full)
            else again = true;
        }
        const unsigned m = __ballot_sync(0xffffffffu, again);
        if (again) {
            const uint32_t at = out + __popc(m & ((1u << lane) - 1));
            q.key[at] = key;
            q.skip[at] = (uint8_t)(skip + 2);
        }
        out += __popc(m);
    }
    __syncwarp();
    q.n = out;
}

// Geometry of a warp tile of kWarpTile window starts for one k.
template <int K>
struct TileGeom {
    static constexpr int Q = 8 * ((K + 7 + 7) / 8);  // bytes a thread pulls per strand
    static constexpr int BL = ((kWarpTile - 8 + Q) + 15) / 16 * 16;
    static constexpr int NV = BL / 16;
    static constexpr int NX = Q / 8;
    static constexpr int NW = (K + 7) / 8;
    static constexpr int NE = BL / 32 + 3;
    static constexpr uint64_t MK = (K == 64) ? ~0ULL : ((1ULL << K) - 1);
    static constexpr uint64_t MK1 = (1ULL << (K - 1)) - 1;
    static constexpr uint64_t TAILMASK = (K % 8) ? (~0ULL >> (8 * (8 - K % 8))) : ~0ULL;
};

// Which of the lane's kWPT consecutive windows (starting at tile-relative position lane * kWPT)
// are counted: inside [w_lo, w_hi), no bad bit in [p, p+K), no end bit in [p, p+K-1).  In the
// error-mode pre-scan (MODE == kModeFirstBad) nothing is valid; the smallest in-read window
// holding a bad byte goes to first_bad instead.
template <int K, int MODE>
__device__ __forceinline__ uint32_t lane_valid_mask(const ConsumeParams &p, const uint16_t *s_bad, const uint32_t *s_end,
                                                    uint64_t w0, int lane, uint64_t &first_bad) {
    constexpr uint64_t MK = TileGeom<K>::MK, MK1 = TileGeom<K>::MK1;
    const int p0 = lane * kWPT;
    const uint32_t *bad32 = reinterpret_cast<const uint32_t *>(s_bad);
    const int wi = p0 >> 5, sh = p0 & 31;
    // bits [p0, p0 + 7 + K) of the two masks: two 32-bit words hold them up to K = 33,
    // three up to K = 64 (sh is 0, 8, 16 or 24)
    const uint64_t mb = (((uint64_t)bad32[wi + 1] << 32) | bad32[wi]) >> sh;
    const uint64_t me = (((uint64_t)s_end[wi + 1] << 32) | s_end[wi]) >> sh;
    uint64_t mb_hi = 0, me_hi = 0;  // bits 64.. of the same, K > 33 only
    if constexpr (K > 33) {
        mb_hi = ((uint64_t)bad32[wi + 2] << 32) >> sh;  // its bit i is mask bit 32 + i
        me_hi = ((uint64_t)s_end[wi + 2] << 32) >> sh;
    }
    const uint64_t gp0 = w0 + p0;

    uint32_t valid = 0;
#pragma unroll
    for (int j = 0; j < kWPT; ++j) {
        const bool in_range = gp0 + j >= p.w_lo && gp0 + j < p.w_hi;
        uint64_t vb = mb >> j, ve = me >> j;
        if constexpr (K > 33) {
            // mask bits [j, j + 64): the low 64 - sh come from the first two words, the rest
            // from the third, whose bit i is mask bit 32 + i
            vb = (mb | (mb_hi << 32)) >> j | (j ? (mb_hi >> 32) << (64 - j) : 0);
            ve = (me | (me_hi << 32)) >> j | (j ? (me_hi >> 32) << (64 - j) : 0);
        }
        const bool in_read = (ve & MK1) == 0;
        const bool clean = (vb & MK) == 0;
        if (MODE == kModeFirstBad) {
            if (in_range && in_read && !clean && gp0 + j + K <= p.data_end)
                first_bad = min(first_bad, gp0 + j);
        } else if (in_range && in_read && clean) {
            valid |= 1u << j;
        }
    }
    return valid;
}

// Hashes of the lane's valid windows (h[j] stays 0 for the others): canonical strand, then
// murmur3 x64_128 seed 42 h1 over its K upper-case ASCII bytes.
template <int K>
__device__ __forceinline__ void lane_hashes(const uint8_t *s_fw, const uint8_t *s_rc, int p0, uint32_t valid,
                                            uint64_t (&h)[kWPT]) {
    constexpr int Q = TileGeom<K>::Q, BL = TileGeom<K>::BL, NX = TileGeom<K>::NX, NW = TileGeom<K>::NW;
    constexpr uint64_t TAILMASK = TileGeom<K>::TAILMASK;
    uint64_t F[NX], R[NX];
    const uint64_t *f64 = reinterpret_cast<const uint64_t *>(s_fw + p0);
    const uint64_t *r64 = reinterpret_cast<const uint64_t *>(s_rc + BL - p0 - Q);
#pragma unroll
    for (int i = 0; i < NX; ++i) { F[i] = f64[i]; R[i] = r64[i]; }

    // Straight-line code for all 8 windows (no branch inside, so the compiler can
    // interleave the independent murmur chains): the strand is chosen from the
    // byte-swapped leading word; a tie on those 8 bases (probability 4^-8 on random
    // sequence) is only recorded here and resolved after the block.
    uint32_t ties = 0;
    auto hash_one = [&](auto jc) {
        constexpr int j = decltype(jc)::value;
        constexpr int FO = j, RO = Q - K - j;
        uint64_t a[NW], b[NW];
        static_for<NW>([&](auto ic) {
            constexpr int i = decltype(ic)::value;
            a[i] = word_at<FO + 8 * i>(F);
            b[i] = word_at<RO + 8 * i>(R);
        });
        a[NW - 1] &= TAILMASK;
        b[NW - 1] &= TAILMASK;
        const bool use_rc = bswap64(b[0]) < bswap64(a[0]);
        if (NW > 1) ties |= (uint32_t)(a[0] == b[0]) << j;
        uint64_t w[NW];
#pragma unroll
        for (int i = 0; i < NW; ++i) w[i] = use_rc ? b[i] : a[i];
        h[j] = ((valid >> j) & 1u) ? murmur_words<K>(w) : 0;
    };
    static_for<kWPT>(hash_one);
    ties &= valid;
    if (NW > 1 && ties) {
        // rare: compare the full k-mers byte by byte from shared memory and redo the hash
        for (int j = 0; j < kWPT; ++j) {
            if (!((ties >> j) & 1u)) continue;
            const uint8_t *fw = s_fw + p0 + j, *rc = s_rc + BL - K - p0 - j;
            bool use_rc = false;
            for (int i = 8; i < K; ++i)
                if (fw[i] != rc[i]) { use_rc = rc[i] < fw[i]; break; }
            const uint8_t *src = use_rc ? rc : fw;
            const uint64_t hv = murmur_bytes([&](int i) -> uint64_t { return src[i]; }, K);
#pragma unroll
            for (int q = 0; q < kWPT; ++q) if (q == j) h[q] = hv;
        }
    }
}

// Specialised kernel (k <= 32).  Every warp is an independent worker: it pulls
// tiles of kWarpTile = 256 window starts from an atomic counter, stages them in
// its private slice of shared memory and only ever executes __syncwarp().  (A
// first version used 2048-window CTA tiles; ncu showed 30 % of all stall samples
// at the CTA barrier waiting for the one warp stuck in a long probe.)
template <int K, int MODE>
__global__ void __launch_bounds__(kThreads, K > 32 ? 2 : OXG_MIN_CTAS) consume_kernel(const ConsumeParams p) {
    static_assert(K >= 1 && K <= 64, "specialised kernel covers k <= 64");
    constexpr int BL = TileGeom<K>::BL, NV = TileGeom<K>::NV, NE = TileGeom<K>::NE;
    constexpr bool kCounts = MODE == kModeCount;
    constexpr int kWarps = kThreads / 32;
    static_assert(NV <= 32 && NE <= 32, "one lane per staged vector / mask word");

    __shared__ __align__(16) uint8_t s_fw_all[kWarps][BL];
    __shared__ __align__(16) uint8_t s_rc_all[kWarps][BL];
    __shared__ __align__(8) uint16_t s_bad_all[kWarps][NV + 6 + ((NV + 6) & 1) + 2];
    __shared__ __align__(8) uint32_t s_end_all[kWarps][NE + (NE & 1)];
    // software pipeline: the next tile's bytes and read boundaries are fetched with cp.async
    // while the current tile is hashed, so no warp waits on a tile's first loads
    __shared__ __align__(16) uint8_t s_raw_all[kWarps][2][BL];
    __shared__ __align__(8) uint64_t s_off_all[kWarps][2][32];
    // dynamic shared memory (see consume_dyn_smem): per warp the slow queue (keys + skip
    // bytes) when counting
    extern __shared__ __align__(16) uint8_t dyn_smem[];
    constexpr int kDynPerWarp = kQueueCap * 9;

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t *s_fw = s_fw_all[warp], *s_rc = s_rc_all[warp];
    uint16_t *s_bad = s_bad_all[warp];
    uint32_t *s_end = s_end_all[warp];
    uint64_t n_counted = 0;
    uint64_t first_bad = ~0ULL;

    uint8_t *dyn = dyn_smem + (kCounts ? warp * kDynPerWarp : 0);
    SlowQueue queue{reinterpret_cast<uint64_t *>(dyn), dyn + kQueueCap * 8, 0};
    uint32_t created = 0;
    bool late = false;  // working on the last quarter of the launch's tiles
    auto flush_created = [&]() {
        const uint32_t tot = __reduce_add_sync(0xffffffffu, created);
        if (lane == 0 && tot) {
            atomicAdd((unsigned long long *)&p.table.ctrl->size, (unsigned long long)tot);
            if (late) atomicAdd((unsigned long long *)&p.table.ctrl->late_new, (unsigned long long)tot);
        }
        created = 0;
    };
    bool tiles_left = true;

    const uint64_t stream_policy = l2_evict_first_policy();
#if OXG_BULK_STAGE
    // one transaction barrier per raw buffer of this warp; a phase = one tile's bytes
    __shared__ __align__(8) uint64_t s_bar_all[kWarps][2];
    uint64_t *s_bar = s_bar_all[warp];
    uint32_t bar_parity = 0;  // bit b: parity to wait for on buffer b
    if (lane == 0) { mbar_init(&s_bar[0], 1); mbar_init(&s_bar[1], 1); mbar_fence_init(); }
    __syncwarp();
    // Bytes past data_end are masked as bad whatever they hold (stage16_raw), so a tile at the
    // end of the data copies whole 16-byte units (at most 15 bytes past the end, inside the
    // same aligned unit as the last base) and leaves the rest of the buffer as it was.
    auto prefetch_raw = [&](uint64_t tile, uint8_t *dst, int b) {
        if (lane == 0) {
            const uint64_t g = p.tile_base + tile * kWarpTile;
            const uint32_t n = g >= p.data_end ? 0u : (uint32_t)min((uint64_t)BL, (uint64_t)((p.data_end - g + 15) & ~15ull));
            mbar_arrive_expect_tx(&s_bar[b], n);
            if (n) bulk_g2s(dst, p.bases + (g - p.g0), n, &s_bar[b], stream_policy);
        }
    };
#else
    auto prefetch_raw = [&](uint64_t tile, uint8_t *dst, int) {
        if (lane < NV) {
            const uint64_t g = p.tile_base + tile * kWarpTile + 16ull * lane;
            const uint32_t n = g >= p.data_end ? 0u : (uint32_t)min((uint64_t)16, p.data_end - g);
            cp_async16_zfill(dst + 16 * lane, n ? p.bases + (g - p.g0) : p.bases, n, stream_policy);
        }
    };
#endif
    auto prefetch_offsets = [&](uint64_t first, uint64_t *dst) {
        const uint64_t r = first + lane;
        if (r < p.n_off) cp_async8(dst + lane, p.offsets + r);
        else dst[lane] = ~0ULL;
    };
    // Tile ids come from one global counter, kTileBatch consecutive tiles per atomic; the
    // request for the next batch is issued when a batch is opened, so its (serialised, one
    // hot address for all warps) latency is hidden behind eight tiles of work.
    uint64_t batch_pos = 0, batch_end = 0, batch_pending = 0;
    auto request_batch = [&]() {
        if (lane == 0) batch_pending = atomicAdd((unsigned long long *)&p.table.ctrl->tile_counter, (unsigned long long)kTileBatch);
    };
    auto next_tile_id = [&]() {
        if (batch_pos == batch_end) {
            batch_pos = __shfl_sync(0xffffffffu, batch_pending, 0);
            batch_end = batch_pos + kTileBatch;
            request_batch();
        }
        return batch_pos++;
    };
    request_batch();
    uint64_t t_cur = next_tile_id(), t_nxt = next_tile_id();
    int buf = 0;
    if (t_cur < p.n_tiles) {
        prefetch_raw(t_cur, s_raw_all[warp][0], 0);
        prefetch_offsets(p.tile_first[t_cur], s_off_all[warp][0]);
    }
    cp_async_commit();

    while (tiles_left) {
        const uint64_t t = t_cur;
        if (t >= p.n_tiles) { tiles_left = false; cp_async_wait<0>(); continue; }
        const uint64_t w0 = p.tile_base + t * kWarpTile;
        late = t * 4 >= p.n_tiles * 3;
        if (MODE == kModeFirstBad && w0 > __ldcg(&p.table.ctrl->first_bad)) {
            // a bad window before this tile is already known: nothing later can be the first
#if OXG_BULK_STAGE
            mbar_wait(&s_bar[buf], (bar_parity >> buf) & 1u);  // this tile's copy is in flight: let it land
#endif
            tiles_left = false; cp_async_wait<0>(); continue;
        }
        uint8_t *s_raw = s_raw_all[warp][buf];
        const uint64_t *s_off = s_off_all[warp][buf];

        // start on the tile after this one: its id is known already, its bytes go to the
        // other half of the raw buffer; the id of the tile after that is requested now
        uint64_t tf_next = 0;
        if (t_nxt < p.n_tiles) {
            tf_next = __ldg(p.tile_first + t_nxt);
            prefetch_raw(t_nxt, s_raw_all[warp][buf ^ 1], buf ^ 1);
        }
        cp_async_commit();
        cp_async_wait<1>();  // everything issued before this iteration (this tile's bytes and boundaries) has landed
#if OXG_BULK_STAGE
        mbar_wait(&s_bar[buf], (bar_parity >> buf) & 1u);
        bar_parity ^= 1u << buf;
#endif
        if (lane < NE) s_end[lane] = 0;
        __syncwarp();

        if (lane < NV) stage16_raw<BL>(p, w0, lane, *reinterpret_cast<const uint4 *>(s_raw + 16 * lane), s_fw, s_rc, s_bad);
        {
            const uint64_t e = s_off[lane] - 1 - w0;  // last base of a read, tile-relative (sentinel: huge)
            if (e < (uint64_t)BL) atomicOr(&s_end[e >> 5], 1u << (e & 31));
            if (__shfl_sync(0xffffffffu, e < (uint64_t)BL, 31)) {
                // more than 32 read boundaries inside one tile (tiny or empty reads): walk the rest
                for (uint64_t r = p.tile_first[t] + 32 + lane; r < p.n_off; r += 32) {
                    const uint64_t e2 = p.offsets[r] - 1 - w0;
                    if (e2 >= (uint64_t)BL) break;
                    atomicOr(&s_end[e2 >> 5], 1u << (e2 & 31));
                }
            }
        }
        bool full = false;
        if (kCounts) full = __ldcg(&p.table.ctrl->size) >= p.table.limit;
        __syncwarp();

        const int p0 = lane * kWPT;
        const uint64_t gp0 = w0 + p0;
        const uint32_t valid = lane_valid_mask<K, MODE>(p, s_bad, s_end, w0, lane, first_bad);

        if (MODE != kModeFirstBad) {
            uint64_t h[kWPT] = {};
            if (valid) lane_hashes<K>(s_fw, s_rc, p0, valid, h);

            // the next tile's read boundaries (its tile_first entry has arrived by now)
            if (t_nxt < p.n_tiles) prefetch_offsets(tf_next, s_off_all[warp][buf ^ 1]);
            cp_async_commit();

            if (MODE == kModeHash) {
#pragma unroll
                for (int j = 0; j < kWPT; ++j)
                    if (gp0 + j >= p.w_lo && gp0 + j < p.w_hi) p.hashes_out[gp0 + j - p.w_lo] = h[j];
            } else if (kCounts) {
                // Warp-aggregated pre-reduction of duplicate hashes, for the pattern that ruins a
                // RED-per-window scheme: low-complexity sequence (homopolymers, short tandem
                // repeats), where a lane's eight windows are a handful of k-mers over and over
                // and every lane of the tile holds the same ones.  A lane that finds one of its
                // hashes at least twice among its eight pools the occurrences with the lanes of
                // the warp that hold the same hash; one of them makes a single update.  Ordinary
                // sequence leaves after eight comparisons.
                for (int round = 0; round < 4; ++round) {
                    uint64_t hv = 0;
#pragma unroll
                    for (int j = kWPT - 1; j >= 0; --j) hv = h[j] != 0 ? h[j] : hv;  // first hash still to count
                    uint32_t same = 0;
#pragma unroll
                    for (int j = 0; j < kWPT; ++j) same |= (uint32_t)(hv != 0 && h[j] == hv) << j;
                    if (__popc(same) < 2) break;
                    const unsigned peers = __match_any_sync(__activemask(), hv);
                    const uint32_t occurrences = __reduce_add_sync(peers, (uint32_t)__popc(same));
                    if (lane == __ffs(peers) - 1) created += table_add(p.table, hv, occurrences, full);
                    n_counted += __popc(same);
#pragma unroll
                    for (int j = 0; j < kWPT; ++j) h[j] = ((same >> j) & 1u) ? 0 : h[j];
                }
                while (queue.n > kQueueCap - kWPT * 32) slow_round(p.table, queue, full, created);
                count_fast8(p.table, h, queue, n_counted);
                slow_round(p.table, queue, full, created);
                flush_created();
            }
        }
        if (MODE == kModeFirstBad) {
            if (t_nxt < p.n_tiles) prefetch_offsets(tf_next, s_off_all[warp][buf ^ 1]);
            cp_async_commit();
        }
        __syncwarp();  // this warp's shared slice is reused by its next tile
        t_cur = t_nxt;
        t_nxt = next_tile_id();
        buf ^= 1;
    }

    if (kCounts) {
        while (queue.n) slow_round(p.table, queue, __ldcg(&p.table.ctrl->size) >= p.table.limit, created);
        flush_created();
    }
    if (MODE == kModeFirstBad) {
        for (int o = 16; o; o >>= 1) first_bad = min(first_bad, __shfl_xor_sync(0xffffffffu, first_bad, o));
        if (lane == 0 && first_bad != ~0ULL)
            atomicMin((unsigned long long *)&p.table.ctrl->first_bad, (unsigned long long)first_bad);
    } else if (kCounts) {
        for (int o = 16; o; o >>= 1) n_counted += __shfl_xor_sync(0xffffffffu, n_counted, o);
        if (lane == 0 && n_counted)
            atomicAdd((unsigned long long *)&p.table.ctrl->counted, (unsigned long long)n_counted);
    }
}

// ---- any k in 1..255: one window per thread, bytes read from shared memory ----
__device__ __forceinline__ uint32_t comp1(uint32_t c) { return c ^ ((c & 2) ? 0x04u : 0x15u); }

template <int MODE>
__global__ void __launch_bounds__(kThreads) consume_generic_kernel(const ConsumeParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int K = (int)p.ksize;
    const int BL = (kTileW + K - 1 + 15) / 16 * 16;
    const int NV = BL / 16;
    uint8_t *s_fw = smem;  // the reverse strand is derived on the fly here
    uint16_t *s_bad = reinterpret_cast<uint16_t *>(smem + BL);
    uint32_t *s_end = reinterpret_cast<uint32_t *>(smem + BL + ((NV * 2 + 15) / 16 * 16) + 16);
    const uint32_t *bad32 = reinterpret_cast<const uint32_t *>(s_bad);

    const int tid = threadIdx.x;
    uint64_t n_counted = 0, first_bad = ~0ULL;

    __shared__ uint64_t s_tile;
    for (;;) {
        if (tid == 0) s_tile = atomicAdd((unsigned long long *)&p.table.ctrl->tile_counter, 1ULL);
        for (int i = tid; i < BL / 32 + 3; i += kThreads) s_end[i] = 0;
        if (tid < 8) s_bad[NV + tid] = 0xffff;
        __syncthreads();
        const uint64_t t = s_tile;
        if (t >= p.n_tiles) break;
        const uint64_t w0 = p.tile_base + t * kTileW;
        for (int v = tid; v < NV; v += kThreads) {
            // same staging as the specialised kernel, BL known only at run time
            const uint64_t g = w0 + 16ull * v;
            uint4 raw = load_bases16(p, g);
            uint32_t u[4] = {upper4(raw.x), upper4(raw.y), upper4(raw.z), upper4(raw.w)};
            uint32_t ok = acgt_mask4(u[0]) | (acgt_mask4(u[1]) << 4) | (acgt_mask4(u[2]) << 8) |
                          (acgt_mask4(u[3]) << 12);
            if (g + 16 > p.data_end)
                ok &= g >= p.data_end ? 0u : (0xffffu >> (16 - (uint32_t)(p.data_end - g)));
            *reinterpret_cast<uint4 *>(s_fw + 16 * v) = make_uint4(u[0], u[1], u[2], u[3]);
            s_bad[v] = (uint16_t)(~ok);
        }
        for (uint64_t r = p.tile_first[t] + tid; r < p.n_off; r += kThreads) {
            const uint64_t e = p.offsets[r] - 1 - w0;
            if (e >= (uint64_t)BL) break;
            atomicOr(&s_end[e >> 5], 1u << (e & 31));
        }
        bool full = false;
        if (MODE == kModeCount) full = __ldcg(&p.table.ctrl->size) >= p.table.limit;
        __syncthreads();

        uint32_t created = 0;
        for (int q = tid; q < kTileW; q += kThreads) {
            const uint64_t gp = w0 + q;
            const bool in_range = gp >= p.w_lo && gp < p.w_hi;
            // any bad bit in [q, q+K), any end bit in [q, q+K-1)
            bool clean = true, in_read = true;
            for (int b = q; b < q + K; ) {
                const int word = b >> 5, off = b & 31;
                const int take = min(32 - off, q + K - b);
                const uint32_t m = (take == 32 ? ~0u : ((1u << take) - 1)) << off;
                if (bad32[word] & m) clean = false;
                const int take_e = min(take, q + K - 1 - b);
                if (take_e > 0) {
                    const uint32_t me = (take_e == 32 ? ~0u : ((1u << take_e) - 1)) << off;
                    if (s_end[word] & me) in_read = false;
                }
                b += take;
            }
            uint64_t h = 0;
            if (MODE == kModeFirstBad) {
                if (in_range && in_read && !clean && gp + K <= p.data_end) first_bad = min(first_bad, gp);
                continue;
            }
            if (in_range && in_read && clean) {
                bool use_rc = false;
                for (int i = 0; i < K; ++i) {
                    const uint32_t a = s_fw[q + i], b = comp1(s_fw[q + K - 1 - i]);
                    if (a != b) { use_rc = b < a; break; }
                }
                h = murmur_bytes(
                    [&](int i) -> uint64_t {
                        return use_rc ? comp1(s_fw[q + K - 1 - i]) : (uint32_t)s_fw[q + i];
                    },
                    K);
            }
            if (MODE == kModeHash) {
                if (in_range) p.hashes_out[gp - p.w_lo] = h;
            } else if (MODE == kModeCount) {
                if (h != 0) { ++n_counted; created += table_add(p.table, h, 1, full); }
            }
        }
        if (MODE == kModeCount) {
            const uint32_t tot = __reduce_add_sync(0xffffffffu, created);
            if ((tid & 31) == 0 && tot) {
                atomicAdd((unsigned long long *)&p.table.ctrl->size, (unsigned long long)tot);
                if (t * 4 >= p.n_tiles * 3) atomicAdd((unsigned long long *)&p.table.ctrl->late_new, (unsigned long long)tot);
            }
        }
        __syncthreads();
    }
    if (MODE == kModeFirstBad) {
        for (int o = 16; o; o >>= 1) first_bad = min(first_bad, __shfl_xor_sync(0xffffffffu, first_bad, o));
        if ((tid & 31) == 0 && first_bad != ~0ULL)
            atomicMin((unsigned long long *)&p.table.ctrl->first_bad, (unsigned long long)first_bad);
    } else if (MODE == kModeCount) {
        for (int o = 16; o; o >>= 1) n_counted += __shfl_xor_sync(0xffffffffu, n_counted, o);
        if ((tid & 31) == 0 && n_counted)
            atomicAdd((unsigned long long *)&p.table.ctrl->counted, (unsigned long long)n_counted);
    }
}

}  // namespace oxg

namespace oxg {
inline size_t generic_smem_bytes(int k) {
    const int BL = (kTileW + k - 1 + 15) / 16 * 16, NV = BL / 16;
    return (size_t)BL + ((NV * 2 + 15) / 16 * 16) + 16 + (BL / 32 + 3) * 4;
}
}  // namespace oxg

namespace oxg {
// dynamic shared memory a specialised consume launch needs
inline size_t consume_dyn_smem(int mode) {
    if (mode != kModeCount) return 0;
    return (size_t)(kThreads / 32) * (kQueueCap * 9);
}
}  // namespace oxg
