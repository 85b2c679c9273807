// scatter.cuh -- pass A of the partitioned pipeline: hash the reads, scatter every hash into
// the fragment of its destination (see aggregate.cuh for pass B and for why).
//
// Replaces the first half of the hot loop of KmerCountTable::consume
// (/root/reference/src/lib.rs:576-600: the SeqToHashes step); the `count_hash` half happens in
// pass B.  Validity, canonical strand and hashing are the device functions of consume.cuh.
//
// What shapes this kernel is the store side.  A scattered store -- one lane, one sector --
// costs a B200 SM about seven cycles whatever its width (8, 16 or 32 bytes: 40 G stores/s
// chip-wide, profiles/r2_microbench_smem_scatter.txt), so "one 8-byte store per hash straight
// into the destination's fragment" runs at a third of the hashing rate.  Shared-memory atomics
// and stores, in contrast, cost 0.13-0.45 cycles.  So a CTA sorts a large batch of hashes by
// destination in shared memory first; a destination's run of the sorted batch then leaves the
// SM as consecutive lanes storing consecutive entries of its fragment.
//
// A CTA is persistent and works in batches of `batch_tiles` warp tiles (256 window starts, 8 per
// lane) per warp:
//   1. hash:      every warp hashes its tiles with no CTA barrier into its own slice of the batch
//                 buffer and counts the hashes per destination (one shared-memory atomic each)
//                                                                                   | barrier
//   2. scan:      one warp per 256 destinations turns the counts into the run start of every
//                 destination in the sorted batch and the offset from there to its fragment's fill
//                 position; every warp loads its slice into registers              | barrier
//   3. permute:   every hash goes to its destination's run, start + atomicAdd(cursor)  | barrier
//   4. write out: warps stride over the sorted batch; the entry at rank r of its run goes to
//                 position fill + r of its fragment, or to the spill list when that is past
//                 frag_cap                                                          | barrier
// The destination is recomputed from the hash wherever it is needed (one multiply and a shift),
// never stored; order within a run is whatever the atomics made it (pass B adds commutatively).
// At the end of a launch frag_cnt holds the fill counts exactly, and a later launch can continue
// the same fragments (frag_append): pass B then runs once per several launches and sees more
// duplicates per key.
// A fragment is [dest][cta][frag_cap] as pass B expects; what does not fit a fragment (skew: one
// k-mer flooding its partition) goes to the spill list exactly as before.
#pragma once
#include "consume.cuh"

namespace oxg {

// Two CTAs of 12 warps per SM rather than one of 24.  One CTA of 24 warps sorts twice the batch
// (18432 hashes) per set of barriers and ran pass A 1 ms faster on C2 (18.7 against 19.7 ms per
// step, one B200) -- but it halves the pass A grid, i.e. the fragments of a partition, and pass B
// then took 9.6 instead of 8.1 ms: the C2 step was 28.6 ms against 28.0 (DESIGN.md 4.3).
#ifndef OXG_SCAT_THREADS
#define OXG_SCAT_THREADS 384
#endif
#ifndef OXG_SCAT_CTAS
#define OXG_SCAT_CTAS 2
#endif
constexpr int kScatThreads = OXG_SCAT_THREADS;
constexpr int kScatCtasPerSm = OXG_SCAT_CTAS;
constexpr int kScatWarps = kScatThreads / 32;
// Warp tiles per warp and batch, at most: step 3 holds a warp's whole slice in registers, 8 hashes
// per lane and tile, and 80 registers per thread (two CTAs of 384 or one of 768 per SM) leave room
// for three tiles' 24 hashes and no more.
constexpr int kScatMaxBatchTiles = 3;
static_assert(kScatWarps * 256 >= 2048, "step 2 scans 256 destinations per warp, up to 2048 of them");

// per-warp tile buffers: forward bytes, mirrored complement, bad bits, end bits
template <int K>
struct ScatWarpBuf {
    static constexpr int BL = TileGeom<K>::BL;
    static constexpr int kBytes = 2 * BL + 64 + 64;
};

// dynamic shared memory: the batch buffer, three words per destination (count, run position,
// fragment-minus-batch offset), the batch total and launch tally, the per-warp tile buffers
__host__ __device__ inline size_t scatter_dest_bytes(uint32_t n_dest) { return ((size_t)n_dest * 12 + 15) & ~(size_t)15; }
__host__ __device__ inline size_t scatter_smem_bytes(uint32_t n_dest, uint32_t batch_tiles, int warp_buf_bytes) {
    return (size_t)kScatWarps * batch_tiles * kWarpTile * 8 + scatter_dest_bytes(n_dest) + 16 + (size_t)kScatWarps * warp_buf_bytes;
}

template <int K>
__global__ void __launch_bounds__(kScatThreads, kScatCtasPerSm) scatter_kernel(const ConsumeParams p) {
    using G = TileGeom<K>;
    constexpr int BL = G::BL, NV = G::NV, NE = G::NE;
    constexpr int kMaxPerLane = kScatMaxBatchTiles * kWPT;
    static_assert(NV + 8 <= 32 && NE <= 16, "per-warp mask buffers are 64 bytes each");
    extern __shared__ __align__(128) uint8_t sm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t nd = p.n_dest, slice = p.batch_tiles * kWarpTile;  // entries of a warp's slice
    uint64_t *batch = reinterpret_cast<uint64_t *>(sm);               // [kScatWarps][slice], then sorted
    // Per destination: cnt = entries of the batch; pos = run start in the sorted batch, after step 3
    // the run's end; to_frag = fragment position minus batch position of the run (mod 2^32).  The
    // fill count of the fragment is never stored: before a batch's scan it is
    // min(to_frag + pos, frag_cap) -- the previous batch's fill plus its run, or where the launch began.
    uint32_t *cnt = reinterpret_cast<uint32_t *>(batch + (size_t)kScatWarps * slice);
    uint32_t *pos = cnt + nd, *to_frag = pos + nd;
    uint32_t *s_total = reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(cnt) + scatter_dest_bytes(nd));  // entries of the batch
    unsigned long long *s_counted = reinterpret_cast<unsigned long long *>(s_total + 2);  // ... of the launch so far
    uint8_t *wbuf = reinterpret_cast<uint8_t *>(s_total + 4) + (size_t)warp * ScatWarpBuf<K>::kBytes;
    uint8_t *s_fw = wbuf, *s_rc = wbuf + BL;
    uint16_t *s_bad = reinterpret_cast<uint16_t *>(wbuf + 2 * BL);
    uint32_t *s_end = reinterpret_cast<uint32_t *>(wbuf + 2 * BL + 64);
    uint64_t *const my_slice = batch + (size_t)warp * slice;

    // (the fragment buffer holds fewer than 2^32 entries: plan_partitioned)
    const uint32_t frag_row = gridDim.x * p.frag_cap;                        // entries between destinations
    uint64_t *const my_frag = p.frag + (uint64_t)blockIdx.x * p.frag_cap;    // + dest * frag_row
    // A launch may continue fragments an earlier launch began (frag_append) at their fill counts.
    for (uint32_t i = threadIdx.x; i < nd; i += kScatThreads) {
        to_frag[i] = p.frag_append ? p.frag_cnt[(uint64_t)i * gridDim.x + blockIdx.x] : 0u;
        cnt[i] = 0; pos[i] = 0;
    }
    if (threadIdx.x == 0) *s_counted = 0;
    __syncthreads();

    auto dest_of = [&](uint64_t h) {
        uint32_t d = (uint32_t)((h * kPhi) >> p.part_shift);
        if (p.n_ranks > 1) d += (uint32_t)(h >> p.owner_shift) * p.n_parts;
        return d;
    };

    uint64_t first_bad_unused = ~0ULL;
    // tile numbers in 32 bits (launch_part_a: fewer than 2^31 tiles), so that they cost the
    // hashing one register each
    const uint32_t n_tiles = (uint32_t)p.n_tiles, tiles_per_round = gridDim.x * kScatWarps;
    const uint32_t n_rounds = (n_tiles + tiles_per_round - 1) / tiles_per_round;
    const uint32_t R = p.batch_tiles, n_batches = (n_rounds + R - 1) / R;  // batch b: rounds [b R, b R + R)
    auto tile_of = [&](uint32_t r) { return (r * gridDim.x + blockIdx.x) * kScatWarps + warp; };

    // software pipeline over tiles: the bytes and read boundaries of the next tile are fetched
    // into registers while this one is hashed
    uint4 raw = make_uint4(0, 0, 0, 0);
    uint64_t tf = 0, off = ~0ULL;
    auto fetch = [&](uint32_t t, uint4 &raw_, uint64_t &tf_) {
        if (t < n_tiles) {
            if (lane < NV) raw_ = load_bases16(p, p.tile_base + (uint64_t)t * kWarpTile + 16ull * lane);
            tf_ = __ldg(p.tile_first + t);
        }
    };
    auto fetch_off = [&](uint32_t t, uint64_t tf_) {
        const uint64_t rr = tf_ + lane;
        return (t < n_tiles && rr < p.n_off) ? __ldg(p.offsets + rr) : ~0ULL;
    };
    fetch(tile_of(0), raw, tf);
    off = fetch_off(tile_of(0), tf);

    for (uint32_t b = 0; b < n_batches; ++b) {
        const uint32_t r0 = b * R, n_here = min(r0 + R, n_rounds) - r0;

        // 1. hash this warp's tiles of the batch into its slice (tile i, window j of lane l at
        //    i * 256 + j * 32 + l; 0 where there is no hash), counting per destination
        for (uint32_t i = 0; i < n_here; ++i) {
            const uint32_t r = r0 + i, t = tile_of(r);
            uint4 raw_next = make_uint4(0, 0, 0, 0);
            uint64_t tf_next = 0;
            fetch(tile_of(r + 1), raw_next, tf_next);
            uint64_t h[kWPT] = {};
            if (t < n_tiles) {
                const uint64_t w0 = p.tile_base + (uint64_t)t * kWarpTile;
                if (lane < NE) s_end[lane] = 0;
                __syncwarp();
                if (lane < NV) stage16_raw<BL>(p, w0, lane, raw, s_fw, s_rc, s_bad);
                {
                    const uint64_t e = off - 1 - w0;  // last base of a read, tile-relative (sentinel: huge)
                    if (e < (uint64_t)BL) atomicOr(&s_end[e >> 5], 1u << (e & 31));
                    if (__shfl_sync(0xffffffffu, e < (uint64_t)BL, 31)) {
                        // more than 32 read boundaries inside one tile (tiny or empty reads): walk the rest
                        for (uint64_t q = tf + 32 + lane; q < p.n_off; q += 32) {
                            const uint64_t e2 = p.offsets[q] - 1 - w0;
                            if (e2 >= (uint64_t)BL) break;
                            atomicOr(&s_end[e2 >> 5], 1u << (e2 & 31));
                        }
                    }
                }
                __syncwarp();
                const uint32_t valid = lane_valid_mask<K, kModePart>(p, s_bad, s_end, w0, lane, first_bad_unused);
                if (valid) lane_hashes<K>(s_fw, s_rc, lane * kWPT, valid, h);
            }
            off = fetch_off(tile_of(r + 1), tf_next);  // its tile_first entry has arrived by now
            raw = raw_next; tf = tf_next;
#pragma unroll
            for (int j = 0; j < kWPT; ++j) {
                // h = 0: a bad window, or the reference's hash==0 skip (src/lib.rs:589)
                if (h[j] != 0) atomicAdd(&cnt[dest_of(h[j])], 1u);
                my_slice[i * kWarpTile + j * 32 + lane] = h[j];
            }
            __syncwarp();  // this warp's tile buffers are restaged by its next tile
        }
        __syncthreads();

        // 2. run starts: an exclusive scan of the counts, warp w taking destinations [256 w, 256 w + 256)
        //    (what lies before them it adds up itself); every warp loads its slice into registers
        if (warp * 256u < nd) {
            const uint32_t lo = warp * 256u;
            uint32_t carry = 0;
            for (uint32_t d = lane; d < lo; d += 32) carry += cnt[d];
            carry = __reduce_add_sync(0xffffffffu, carry);
            uint32_t v[8], x[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const uint32_t d = lo + 32 * u + lane;
                v[u] = d < nd ? cnt[d] : 0u;
                x[u] = v[u];
            }
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const uint32_t y = __shfl_up_sync(0xffffffffu, x[u], o);
                    if (lane >= o) x[u] += y;
                }
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const uint32_t d = lo + 32 * u + lane;
                if (d < nd) {
                    const uint32_t start = carry + x[u] - v[u], fill = min(to_frag[d] + pos[d], p.frag_cap);
                    pos[d] = start; to_frag[d] = fill - start;
                }
                carry += __shfl_sync(0xffffffffu, x[u], 31);
            }
            if (lane == 0 && lo + 256u >= nd) { *s_total = carry; *s_counted += carry; }
        }
        uint64_t v[kMaxPerLane];
#pragma unroll
        for (int u = 0; u < kMaxPerLane; ++u) v[u] = u < (int)(n_here * kWPT) ? my_slice[u * 32 + lane] : 0ull;
        __syncthreads();

        // 3. permute: every hash to its destination's run; the counts are cleared for the next batch
        for (uint32_t d = threadIdx.x; d < nd; d += kScatThreads) cnt[d] = 0;
#pragma unroll
        for (int u = 0; u < kMaxPerLane; ++u)
            if (v[u] != 0) batch[atomicAdd(&pos[dest_of(v[u])], 1u)] = v[u];
        __syncthreads();

        // 4. write out: consecutive lanes store consecutive entries of a run; four chunks of 32
        //    entries per warp at a time, so that the loads and stores of one do not wait for another's
        const uint32_t total = *s_total;
        for (uint32_t i0 = warp * 128; i0 < total; i0 += kScatThreads * 4) {
            uint64_t h[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint32_t i = i0 + 32 * u + lane;
                h[u] = i < total ? batch[i] : 0ull;  // (a sorted entry is never 0)
            }
            uint32_t spilled = 0;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (h[u] == 0) continue;
                const uint32_t d = dest_of(h[u]), at = i0 + 32 * u + lane + to_frag[d];
                if (at < p.frag_cap) my_frag[d * frag_row + at] = h[u];
                else spilled |= 1u << u;
            }
            if (__any_sync(0xffffffffu, spilled != 0)) {
                // skewed input (one k-mer flooding its partition): one reservation per warp and 128 entries
                const uint32_t mine = __popc(spilled);
                uint32_t incl = mine;
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += y;
                }
                unsigned long long base = 0;
                if (lane == 31) base = atomicAdd(p.spill_n, (unsigned long long)incl);
                base = __shfl_sync(0xffffffffu, base, 31) + (incl - mine);
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if ((spilled >> u) & 1u) { if (base < p.spill_cap) p.spill[base] = h[u]; ++base; }
            }
        }
        __syncthreads();
    }

    for (uint32_t d = threadIdx.x; d < nd; d += kScatThreads)
        p.frag_cnt[(uint64_t)d * gridDim.x + blockIdx.x] = min(to_frag[d] + pos[d], p.frag_cap);
    if (threadIdx.x == 0 && *s_counted) atomicAdd((unsigned long long *)&p.table.ctrl->counted, *s_counted);
}

}  // namespace oxg
