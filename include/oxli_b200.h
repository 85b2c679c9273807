/*
 * oxli_b200.h -- C ABI of the B200-native k-mer counting engine.
 *
 * This is the drop-in boundary for the hot path of oxli-bio/oxli
 * (reference: src/lib.rs, one pyo3 class `KmerCountTable`).  Every entry
 * point replaces the Rust/sourmash code behind one group of reference
 * methods; the reference lines each one stands in for are cited below
 * (paths relative to the reference root).  A pyo3 crate would bind these
 * with a plain `extern "C"` block (see INTEGRATION.md); in this repository
 * the host mirror is oxli_b200/csrc/pyoxli.cpp.
 *
 * Conventions
 *   - plain C types only; all sizes are uint64_t; no exceptions cross the ABI.
 *   - every function returns an oxg_status (0 = OK).  oxg_last_error() gives a
 *     thread-local human-readable message for the last non-OK status.
 *   - `oxg_table*` is an opaque handle to a count table living in the HBM of one
 *     GPU.  One handle is used by one caller thread at a time (mirrors the
 *     `&mut self` borrow of the reference, src/lib.rs:41-838).
 *   - pointers named `d_*` are DEVICE pointers on the table's GPU; all other
 *     pointers are HOST pointers (pageable or pinned; pinned avoids a staging
 *     copy, see oxg_pinned_alloc).
 *   - there is no CPU fallback: every call fails with OXG_ERR_CUDA when no
 *     usable sm_100 device is present.
 */
#ifndef OXLI_B200_H
#define OXLI_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum oxg_status {
    OXG_OK = 0,
    OXG_ERR_CUDA = 1,        /* CUDA runtime failure / no device */
    OXG_ERR_INVALID = 2,     /* bad argument */
    OXG_ERR_BAD_KMER = 3,    /* non-ACGT window met in error mode (src/lib.rs:593-596) */
    OXG_ERR_NOMEM = 4,       /* host or device allocation failed */
    OXG_ERR_WRONG_KSIZE = 5, /* k-mer length != table ksize (src/lib.rs:66-67,146-149) */
    OXG_ERR_TOO_SMALL = 6,   /* caller-provided output buffer too small */
    OXG_ERR_IO = 7           /* a file could not be created, opened or written */
} oxg_status;

typedef struct oxg_table oxg_table;

/* thread-local message for the last failing call on this thread */
const char *oxg_last_error(void);
/* library version string; `KmerCountTable.version` (src/lib.rs:27,525-527) */
const char *oxg_version(void);
/* number of visible CUDA devices (0 when none; never fails) */
int oxg_device_count(void);

/* ---- lifecycle: KmerCountTable::new (src/lib.rs:44-62) -------------------
 * ksize in 1..255.  capacity_hint = expected number of distinct k-mers (0 =
 * unknown; the table grows by rehashing on the device). */
oxg_status oxg_table_create(int device, uint32_t ksize, uint64_t capacity_hint, oxg_table **out);
oxg_status oxg_table_destroy(oxg_table *t);
/* drop every entry, keep the allocation */
oxg_status oxg_table_clear(oxg_table *t);
/* make room for `n_keys` distinct keys without further growth */
oxg_status oxg_table_reserve(oxg_table *t, uint64_t n_keys);
oxg_status oxg_table_ksize(const oxg_table *t, uint32_t *ksize);
/* slots currently allocated (16 B each) */
oxg_status oxg_table_capacity(const oxg_table *t, uint64_t *slots);

/* ---- sequence -> hashes: sourmash SeqToHashes(force=true) as driven from
 * src/lib.rs:65-81 (hash_kmer) and 873-881 (kmers_and_hashes) ---------------
 * One hash per window of `seq` (len-k+1 entries, none when len < k); 0 marks a
 * window holding a non-ACGT byte.  Runs the same device code as consume. */
oxg_status oxg_hash_windows(oxg_table *t, const uint8_t *seq, uint64_t len, uint64_t *hashes_out);

/* ---- bulk ingest: KmerCountTable::consume (src/lib.rs:545-607) ------------
 * A batch is a flat byte buffer plus n_reads+1 offsets (CSR); read r is
 * bases[offsets[r] .. offsets[r+1]).  Semantics are those of calling
 * consume(read_r, skip_bad) for r = 0, 1, ... in order:
 *   skip_bad != 0  windows holding a non-ACGT byte are skipped, not counted.
 *   skip_bad == 0  reads before the first read with a bad window are counted in
 *                  full; in that read the windows before the first bad one are
 *                  counted and stay counted; nothing after it is.  The call
 *                  then returns OXG_ERR_BAD_KMER with *err_read = that read and
 *                  *err_pos = the number of its windows counted (the {n} of
 *                  "bad k-mer encountered at position {n}").
 * *total_counted = k-mers added to the table (valid windows whose hash is 0 are
 * skipped and not counted, src/lib.rs:589).  err_read = -1 when no error.
 * The host variant streams the buffer to the GPU in 64 MiB chunks through a ring of
 * four staging buffers (cudaMemcpyAsync on a copy stream, fed by a producer thread, which
 * also checks that the offsets are non-decreasing: on OXG_ERR_INVALID for that reason the
 * table may already hold the reads of earlier chunks). */
oxg_status oxg_consume_batch(oxg_table *t, const uint8_t *bases, const uint64_t *offsets,
                             uint64_t n_reads, int skip_bad, uint64_t *total_counted,
                             int64_t *err_read, uint64_t *err_pos);
/* same, inputs already resident in the table's HBM: d_bases 16-byte aligned, d_offsets[0]
 * must be 0 (the batch is the bytes [0, total_bases)), offsets non-decreasing -- device
 * arrays are not validated */
oxg_status oxg_consume_batch_device(oxg_table *t, const uint8_t *d_bases, const uint64_t *d_offsets,
                                    uint64_t n_reads, uint64_t total_bases, int skip_bad,
                                    uint64_t *total_counted, int64_t *err_read,
                                    uint64_t *err_pos);
/* hash-only pass over a device-resident batch: d_hashes_out[w] for every window
 * start w in [0, total_bases - k + 1) of the flat buffer; 0 for windows that hold
 * a bad byte or straddle two reads.  (First half of the two-kernel pipeline.) */
oxg_status oxg_hash_batch_device(oxg_table *t, const uint8_t *d_bases, const uint64_t *d_offsets,
                                 uint64_t n_reads, uint64_t total_bases, uint64_t *d_hashes_out);

/* ---- increment / lookup by hash (src/lib.rs:100-104, 185-194, 675-681) ---- */
/* counts[h] += 1 for every h; new_counts (nullable) receives the count after
 * each increment (exact for distinct hashes; for duplicates inside one call the
 * values are the counts seen by each increment in some serial order). */
oxg_status oxg_count_hashes(oxg_table *t, const uint64_t *hashes, uint64_t n, uint64_t *new_counts);
/* device-resident list; skip_zero != 0 ignores entries equal to 0 (the hash
 * stream of oxg_hash_batch_device marks uncountable windows with 0);
 * *n_counted (nullable) = increments applied */
oxg_status oxg_count_hashes_device(oxg_table *t, const uint64_t *d_hashes, uint64_t n, int skip_zero,
                                   uint64_t *n_counted);
/* counts[keys[i]] += vals[i], creating keys as needed (a created key may keep the
 * value 0).  Bulk form of count_hash/__setitem__ used by load() (src/lib.rs:297-322). */
oxg_status oxg_add_pairs(oxg_table *t, const uint64_t *keys, const uint64_t *vals, uint64_t n);
/* counts_out[i] = counts.get(hashes[i]).unwrap_or(0), order-preserving */
oxg_status oxg_get_hashes(oxg_table *t, const uint64_t *hashes, uint64_t n, uint64_t *counts_out);
/* counts.insert(h, v): overwrite or create (0 is a legal stored value) */
oxg_status oxg_set_hash(oxg_table *t, uint64_t hash, uint64_t value);
/* counts.remove(h) for each h (src/lib.rs:197-224); *n_removed nullable */
oxg_status oxg_erase_hashes(oxg_table *t, const uint64_t *hashes, uint64_t n, uint64_t *n_removed);
/* mincut (mode 0: remove count < thresh, src/lib.rs:227-246) / maxcut (mode 1:
 * remove count > thresh, src/lib.rs:249-267) */
oxg_status oxg_cut(oxg_table *t, int mode, uint64_t thresh, uint64_t *n_removed);

/* ---- scans: __len__, sum_counts, min, max, histo (src/lib.rs:464-539,665) -- */
typedef struct oxg_stats {
    uint64_t len; /* distinct keys */
    uint64_t sum; /* sum of counts (wrapping u64) */
    uint64_t min; /* 0 when empty */
    uint64_t max; /* 0 when empty */
} oxg_stats;
oxg_status oxg_table_len(oxg_table *t, uint64_t *len);
oxg_status oxg_table_stats(oxg_table *t, oxg_stats *out);
/* histo(zero=False): (freq, n) pairs sorted by freq.  Writes min(*n_out, cap)
 * pairs; call with cap = 0 to size the buffers. */
oxg_status oxg_histo(oxg_table *t, uint64_t *freq, uint64_t *n, uint64_t cap, uint64_t *n_out);

/* order-independent digests of this table (parity checks at sizes where nothing can be
 * exported): out = {len, sum c, xor h, sum h*c mod 2^64, keys whose owner
 * h >> (64 - log2 n_ranks) is not `rank`}; n_ranks = 1, rank = 0 for a plain table */
oxg_status oxg_table_digest(oxg_table *t, int n_ranks, int rank, uint64_t out[5]);

/* ---- export: hashes / dump / __iter__ (src/lib.rs:330-381, 517-521, 658) ---
 * sort_mode 0: table (slot) order -- stable between calls while the table is
 * not modified, so dump() == list(iter); 1: by key; 2: by (count, key). */
oxg_status oxg_export(oxg_table *t, uint64_t *keys, uint64_t *vals, uint64_t cap, int sort_mode,
                      uint64_t *n_out);

/* ---- set comparisons on key sets (src/lib.rs:610-655, 708-722) ------------ */
oxg_status oxg_setop_sizes(oxg_table *a, oxg_table *b, uint64_t *inter, uint64_t *uni);
typedef enum oxg_setop {
    OXG_UNION = 0,
    OXG_INTERSECTION = 1,
    OXG_DIFFERENCE = 2,
    OXG_SYMMETRIC_DIFFERENCE = 3
} oxg_setop;
/* writes min(*n_out, cap) keys (unordered) */
oxg_status oxg_setop_export(oxg_table *a, oxg_table *b, int op, uint64_t *keys_out, uint64_t cap,
                            uint64_t *n_out);
/* n(A&B) / n(A|B) as one IEEE-754 double divide; 1.0 when both are empty */
oxg_status oxg_jaccard(oxg_table *a, oxg_table *b, double *out);
/* cosine similarity of the count vectors (src/lib.rs:727-765) */
oxg_status oxg_cosine(oxg_table *a, oxg_table *b, double *out);

/* ---- merge: KmerCountTable::add (src/lib.rs:778-837) ---------------------- */
oxg_status oxg_merge(oxg_table *dst, oxg_table *src, uint64_t *counts_added, uint64_t *new_keys);

/* ---- hash-sharded table across the GPUs of one node ------------------------
 * The north_star's multi-GPU layout: shard r of N owns the hashes with
 * h >> (64 - log2 N) == r; the reference's primitive for combining partial
 * tables is KmerCountTable::add (src/lib.rs:778-837).  Reads need no such step:
 * consume routes every hash to its owner before it is counted.  Tables counted
 * elsewhere (on one GPU, or another sharded table) are added with
 * oxg_shard_merge_table / oxg_shard_merge below, and keys are removed with
 * oxg_shard_erase_hashes* / oxg_shard_cut.  One oxg_shard per GPU.  The
 * shards of a table live in one process each (the usual arrangement, connected
 * through CUDA IPC handles that the launcher passes around) or in one process
 * together (oxg_shard_connect_local; also how a single-GPU box tests N > 1).
 *
 * Exchange: every rank hashes ITS reads and leaves the hashes in its own HBM,
 * in fragments addressed by (owner, table partition); the owner's aggregation
 * kernel reads the fragments of all ranks through peer-mapped pointers, so the
 * NVLink transfer is that kernel's load stream.  Ranks synchronise through
 * 8-byte flags in each other's exchange header, awaited on the GPU: no host
 * round trip per round, no collective library.
 *
 * oxg_shard_consume_batch* is COLLECTIVE: every rank of the table calls it (with
 * its own reads, possibly none), as are the oxg_shard_* reductions below.  A
 * shard handle is used by one thread at a time; different shards of one process
 * are driven by different threads.  n_ranks: power of two, 1..16; the k must have
 * a specialised kernel (csrc/klist.h).  capacity_hint = distinct keys expected in
 * THIS shard (0 = unknown); round_windows = window starts per rank and exchange
 * round at most (0 = 64 Mi), which fixes the size of the exchange area -- all
 * ranks must pass the same ksize, n_ranks, capacity_hint and round_windows.
 * Larger rounds make larger fragments and a cheaper aggregation (C3, 2 GPUs:
 * 87 / 75 ms per step at 64 / 256 Mi) for about 45 bytes of exchange area per
 * window; a batch from host memory, and a batch into a table that has yet to
 * find its size, run in rounds of 64 Mi at most whatever this says. */
typedef struct oxg_shard oxg_shard;
oxg_status oxg_shard_create(int device, uint32_t ksize, int rank, int n_ranks, uint64_t capacity_hint,
                            uint64_t round_windows, oxg_shard **out);
oxg_status oxg_shard_destroy(oxg_shard *s);
/* the shard's own table: every oxg_table_* / oxg_histo / oxg_export / ... call
 * works on it and sees the keys this rank owns */
oxg_table *oxg_shard_table(oxg_shard *s);
oxg_status oxg_shard_info(const oxg_shard *s, int *rank, int *n_ranks, uint32_t *n_parts,
                          uint64_t *round_windows, uint64_t *exchange_bytes);
/* 64-byte cudaIpcMemHandle_t of this shard's exchange area */
oxg_status oxg_shard_export(oxg_shard *s, uint8_t handle_out[64]);
/* handles = n_ranks * 64 bytes, entry r exported by rank r (entry `rank` ignored) */
oxg_status oxg_shard_connect(oxg_shard *s, const uint8_t *handles);
/* all shards of the table live in this process: shards[i] is rank i of n */
oxg_status oxg_shard_connect_local(oxg_shard *const *shards, int n);
/* KmerCountTable::consume (src/lib.rs:545-607) for this rank's reads, batch form as
 * oxg_consume_batch.  *counted = valid k-mers of THIS rank's reads (what the
 * reference's consume calls would have returned, summed); *absorbed = k-mers counted
 * into this shard (from every rank's reads).  skip_bad == 0: this rank's reads are
 * counted up to its first bad window, and the call returns OXG_ERR_BAD_KMER with
 * err_read / err_pos as in oxg_consume_batch; the other ranks are not affected.
 * The host variant streams the buffer through a ring of staging buffers. */
oxg_status oxg_shard_consume_batch(oxg_shard *s, const uint8_t *bases, const uint64_t *offsets,
                                   uint64_t n_reads, int skip_bad, uint64_t *counted,
                                   uint64_t *absorbed, int64_t *err_read, uint64_t *err_pos);
/* same, inputs resident in this shard's HBM; d_offsets[0] must be 0 and d_bases
 * 16-byte aligned */
oxg_status oxg_shard_consume_batch_device(oxg_shard *s, const uint8_t *d_bases,
                                          const uint64_t *d_offsets, uint64_t n_reads,
                                          uint64_t total_bases, int skip_bad, uint64_t *counted,
                                          uint64_t *absorbed, int64_t *err_read, uint64_t *err_pos);
/* get_hash_array on the whole sharded table (src/lib.rs:185-194), COLLECTIVE: every
 * rank calls it with its own list (n may be 0, and may differ between ranks).
 * counts_out[i] = count of hashes[i] in the table (0 when absent), in the order of
 * the queries.  Any u64 is a legal query: 0, 2^64-1 (its owner's side entry), and
 * duplicates.  Each query goes to the rank that owns it and is answered there: the
 * queries travel in rounds of round_windows per rank, the same exchange rounds a
 * consume call runs, so lookups and consume calls may follow each other in any
 * order.  Plain-table calls on oxg_shard_table(s) made before the call are seen.
 * A call refused for its arguments (null lists with n > 0, an unconnected shard, a
 * device list in another device's memory) returns OXG_ERR_INVALID before it takes
 * part in any exchange. */
oxg_status oxg_shard_get_hashes(oxg_shard *s, const uint64_t *hashes, uint64_t n, uint64_t *counts_out);
/* same, with both lists resident in this shard's HBM */
oxg_status oxg_shard_get_hashes_device(oxg_shard *s, const uint64_t *d_hashes, uint64_t n,
                                       uint64_t *d_counts_out);
/* KmerCountTable::add (src/lib.rs:778-837) into a sharded table, COLLECTIVE: every rank passes its
 * own plain table `src` on this shard's device, or NULL to add nothing.  counts[h] += src[h] for every
 * key of every rank's table: keys held with count 0 are created with 0, 2^64-1 included (its
 * owner's side entry), counts wrap mod 2^64.  src is not modified.  *counts_added and *new_keys
 * (nullable) are totals over the whole table, identical on every rank; new_keys counts, as
 * oxg_merge does, contributions to a key whose count was 0 just before them.  When the same key
 * comes from several ranks in one call, the order of the additions is unspecified: new_keys is
 * then the sum of what adding the ranks' tables one after another would report when no
 * contributed count is 0, and what some serial order would report otherwise.  Each pair travels
 * to the rank that owns its key in exchange rounds of round_windows slots of src, the same rounds
 * consume and lookups run, so all three may follow each other in any order; every owner grows
 * once, before the first round, to hold every key it may receive.  Plain-table calls on src and
 * on oxg_shard_table(dst) made before the call are seen.  Refused before any exchange, with the
 * table unchanged: an unconnected dst, a src on another device or src == oxg_shard_table(dst)
 * (OXG_ERR_INVALID), a different ksize (OXG_ERR_WRONG_KSIZE). */
oxg_status oxg_shard_merge_table(oxg_shard *dst, oxg_table *src, uint64_t *counts_added, uint64_t *new_keys);
/* the same for a sharded src with the same n_ranks, rank and device on every rank: each rank
 * merges src's shard into its own, nothing crosses between GPUs except the two totals.  Also
 * refused (OXG_ERR_INVALID): src == dst, or src sharded another way. */
oxg_status oxg_shard_merge(oxg_shard *dst, oxg_shard *src, uint64_t *counts_added, uint64_t *new_keys);
/* drop_hash for a list on the whole sharded table (src/lib.rs:197-224), COLLECTIVE: every rank
 * passes its own list (n may be 0, and may differ between ranks).  Each hash goes to the rank that
 * owns it, which removes it.  Any u64 is a legal key: 0, duplicates, and 2^64-1 (its owner's side
 * entry); absent keys are ignored.  *n_removed (nullable) = distinct keys removed from the whole
 * table, 2^64-1 included, identical on every rank: a key listed several times, by one rank or by
 * several, counts once.  The keys travel in exchange rounds of round_windows per rank, the same
 * rounds consume, lookups and merges run, so all four may follow each other in any order.  Fewer
 * than 256 keys over all ranks are erased in place, one at a time (the reference's drop /
 * drop_hash); a longer list marks its keys' slots and each owner rebuilds its table once, at the
 * same capacity (the call never grows the table).  Plain-table calls on oxg_shard_table(s) made
 * before the call are seen.  Refused before any exchange, with the table unchanged
 * (OXG_ERR_INVALID): a null list with n > 0, an unconnected shard, a device list outside this
 * shard's device memory.  The slot bitmap (cap / 8 bytes) is reserved before the first exchange
 * too: when that fails the call returns OXG_ERR_NOMEM (OXG_ERR_CUDA for any other CUDA error),
 * again with the table unchanged. */
oxg_status oxg_shard_erase_hashes(oxg_shard *s, const uint64_t *hashes, uint64_t n, uint64_t *n_removed);
/* same, with the list resident in this shard's HBM (left as it was) */
oxg_status oxg_shard_erase_hashes_device(oxg_shard *s, const uint64_t *d_hashes, uint64_t n, uint64_t *n_removed);
/* mincut (mode 0: drop counts < thresh) / maxcut (mode 1: drop counts > thresh) on every shard
 * (src/lib.rs:227-267), COLLECTIVE; *n_removed (nullable) = keys removed from the whole table,
 * 2^64-1 included, identical on every rank.  Refused before any exchange (OXG_ERR_INVALID): an
 * unconnected shard, a mode other than 0 / 1. */
oxg_status oxg_shard_cut(oxg_shard *s, int mode, uint64_t thresh, uint64_t *n_removed);
/* The whole sharded table in one order, each rank holding its own shard's part (hashes /
 * dump / __iter__, src/lib.rs:330-381), COLLECTIVE: every rank passes the same sort_mode, that
 * of oxg_export (0: slot order, 1: by key, 2: by (count, key)).  Every key of rank r is below
 * every key of rank r + 1, so the order of the whole table is each rank's own export placed at
 * the right positions; no pair crosses between GPUs.  keys / vals receive min(*n_out, cap) of this
 * rank's pairs in sort_mode order, 2^64-1 (its owner's side entry) and keys held with count 0
 * included.  runs receives min(*n_runs_out, runs_cap) pieces (global_start, length), 2 u64 each:
 * taken in order they cover keys / vals and say where they go in the whole table.  Modes 0 and 1:
 * one run per rank (the ranks' blocks in rank order); mode 2: one run per distinct count of this
 * rank.  *total_out = pairs in the whole table, the same on every rank.  Output pointers are
 * nullable; call with cap = runs_cap = 0 to size the arrays.  Plain-table calls on
 * oxg_shard_table(s) made before the call are seen.  Refused before any exchange
 * (OXG_ERR_INVALID): an unconnected shard, a bad sort_mode, null arrays with a nonzero cap.  Any
 * other failure on one rank (a device reservation among them, OXG_ERR_NOMEM) reaches every rank in
 * the call's exchange: every rank then returns the status of the first rank that failed. */
oxg_status oxg_shard_export_pairs(oxg_shard *s, int sort_mode, uint64_t *keys, uint64_t *vals, uint64_t cap,
                                  uint64_t *n_out, uint64_t *runs, uint64_t runs_cap, uint64_t *n_runs_out,
                                  uint64_t *total_out);
/* dump(file, sortcounts, sortkeys) of the whole sharded table (src/lib.rs:330-381), COLLECTIVE:
 * every rank passes the same path and sort_mode, and the ranks write ONE file together, the lines
 * "<hash>\t<count>\n" (u64 in decimal) in the order of oxg_shard_export_pairs.  Modes 1 and 2 give
 * the bytes a plain table holding the same pairs dumps; mode 0 the same lines, each rank's in one
 * block, the blocks in rank order.  Each rank sorts and formats its shard on its GPU; rank 0
 * creates the file at its final size, then every rank writes its byte ranges into it.  Refused
 * before any exchange (OXG_ERR_INVALID): an unconnected shard, a bad sort_mode, a null path.  Any
 * other failure on one rank reaches every rank in the call's exchange, and every rank returns the
 * first failing rank's status: ranks that passed different paths (OXG_ERR_INVALID), a device
 * reservation (OXG_ERR_NOMEM), a file that cannot be created, opened or written (OXG_ERR_IO; the
 * file may then be left incomplete). */
oxg_status oxg_shard_dump(oxg_shard *s, const char *path, int sort_mode);
/* time of the last consume call on this shard's stream (device variant: CUDA events;
 * host variant: wall clock of the call) and its number of exchange rounds */
oxg_status oxg_shard_last_ms(const oxg_shard *s, float *ms, uint64_t *rounds);
/* reductions over the whole table (collective; every rank receives the result):
 * len / sum_counts / min / max (src/lib.rs:492-539,665), histo(zero=False)
 * (464-488), |A & B| and |A | B| of two tables sharded the same way (610-638),
 * jaccard (708-722, one f64 divide of the two reduced integers) */
oxg_status oxg_shard_stats(oxg_shard *s, oxg_stats *out);
oxg_status oxg_shard_histo(oxg_shard *s, uint64_t *freq, uint64_t *n, uint64_t cap, uint64_t *n_out);
oxg_status oxg_shard_setop_sizes(oxg_shard *a, oxg_shard *b, uint64_t *inter, uint64_t *uni);
oxg_status oxg_shard_jaccard(oxg_shard *a, oxg_shard *b, double *out);
/* union / intersection / difference / symmetric_difference of two tables sharded the same way
 * (src/lib.rs:610-655), COLLECTIVE: every rank passes the same op (an oxg_setop).  A key is a
 * member when it is present, held with count 0 too.  A key of A owned by rank r can only be in B's
 * shard on rank r, so each rank computes its own part on its GPU and no key crosses between GPUs.
 * keys receives min(*n_out, cap) of the keys of the result that this rank owns, in ascending key
 * order (2^64-1, its owner's side entry, last on the last rank); *start_out (nullable) = the sum of
 * *n_out over the ranks below this one, *total_out (nullable) = the size of the whole result, the
 * same on every rank.  So the parts in rank order are the whole result sorted.  cap >= the lengths
 * of both shard tables of this rank (oxg_table_len on oxg_shard_table, not collective) always
 * suffices.  a == b is allowed.  Plain-table calls on either shard's table made before the call are
 * seen.  Refused before any exchange (OXG_ERR_INVALID), both tables unchanged: a null or
 * unconnected shard, a null n_out, keys == NULL with cap > 0, an op outside 0..3, a and b sharded
 * differently or on different devices.  Any other failure on one rank (ranks that passed different
 * ops: OXG_ERR_INVALID; a device reservation: OXG_ERR_NOMEM) reaches every rank in the call's
 * exchange, and every rank returns the status of the first rank that failed. */
oxg_status oxg_shard_setop_export(oxg_shard *a, oxg_shard *b, int op, uint64_t *keys, uint64_t cap, uint64_t *n_out,
                                  uint64_t *start_out, uint64_t *total_out);
/* cosine similarity of the count vectors of two tables sharded the same way (src/lib.rs:727-765),
 * COLLECTIVE: each rank computes the terms of its shards (dot product as wrapping u64, the sums of
 * squares as doubles, side entries included), one exchange carries them, and every rank sums them
 * in rank order: *out is the same double on every rank.  0.0 when the whole of A or of B is empty
 * or a norm is 0.  Refused before any exchange (OXG_ERR_INVALID) as oxg_shard_setop_export, and
 * for a null out. */
oxg_status oxg_shard_cosine(oxg_shard *a, oxg_shard *b, double *out);
/* order-independent digests of the whole table: out = {len, sum c, xor h,
 * sum h*c mod 2^64, keys found on a rank that does not own them (must be 0)} */
oxg_status oxg_shard_digest(oxg_shard *s, uint64_t out[5]);
/* small all-gather through the exchange headers (collective): every rank gives
 * len <= 1 MiB bytes, out receives n_ranks * len bytes in rank order */
oxg_status oxg_shard_allgather(oxg_shard *s, const void *mine, uint32_t len, void *out);

/* ---- synthetic reads for benchmarks (SURVEY.md section 8d) ----------------
 * Fills d_bases with n_reads reads of read_len bases drawn from a random genome
 * of genome_len bases (counter-based splitmix64; strand flip with p=1/2;
 * substitutions with probability sub_ppm/1e6, N with probability n_ppm/1e6).
 * Read i is a pure function of (seed, first_read + i). */
oxg_status oxg_synth_reads_device(int device, uint8_t *d_bases, uint64_t n_reads, uint32_t read_len,
                                  uint64_t genome_len, uint64_t seed, uint64_t first_read,
                                  uint32_t sub_ppm, uint32_t n_ppm);

/* ---- host helpers ---------------------------------------------------------- */
oxg_status oxg_pinned_alloc(uint64_t bytes, void **out);
oxg_status oxg_pinned_free(void *p);
oxg_status oxg_device_alloc(int device, uint64_t bytes, void **d_out);
oxg_status oxg_device_free(int device, void *d_ptr);
oxg_status oxg_memcpy_h2d(int device, void *d_dst, const void *src, uint64_t bytes);
oxg_status oxg_memcpy_d2h(int device, void *dst, const void *d_src, uint64_t bytes);
/* block until everything queued for this table's GPU has finished */
oxg_status oxg_sync(oxg_table *t);
/* CUDA-event stopwatch on the stream this table's kernels are launched on */
oxg_status oxg_timer_start(oxg_table *t);
oxg_status oxg_timer_stop(oxg_table *t, float *ms);
/* kernels launched by this library in this process so far (bench bookkeeping) */
uint64_t oxg_launch_count(void);
/* CUDA buffers, events and streams the library holds now (tests: what an error return leaves) */
uint64_t oxg_live_allocations(void);
/* tests: the n-th allocation or handle creation of the library from now on fails as if the
 * device were out of memory (OXG_ERR_NOMEM); 0 = none.  Returns the countdown it replaces:
 * 0 once the failure it set has happened (or none was set) */
uint64_t oxg_fail_allocation_after(uint64_t n);
/* device-time of the consume kernels of the last oxg_consume_* call on `t`, in
 * milliseconds, and their number (CUDA events on the launch stream) */
oxg_status oxg_last_consume_kernel_ms(oxg_table *t, float *ms, uint64_t *launches);
/* Process-wide choice of the counting pipeline behind oxg_consume_*: 0 = by launch size
 * (default: launches of >= 8 Mi windows are partitioned), 1 = always the fused
 * hash-and-update kernel, 2 = always the partitioned pipeline (hash + scatter, then
 * aggregate + merge) when the k has a specialised kernel.  n_parts (0 = derived from the
 * table size; else a power of two in 2..8192) and groups (0 = default) are tuning knobs of
 * the partitioned pipeline.  Results are identical whichever is chosen.  Initial values come
 * from OXLI_B200_PIPELINE=fused|part, OXLI_B200_PARTS, OXLI_B200_GROUPS. */
oxg_status oxg_set_pipeline(int choice, uint32_t n_parts, uint32_t groups);
/* of that time, the share of the two passes of the partitioned pipeline (hash + scatter,
 * aggregate + merge); both 0 when the last call ran the fused kernel only */
oxg_status oxg_last_consume_pass_ms(oxg_table *t, float *ms_scatter, float *ms_aggregate);

#ifdef __cplusplus
}
#endif
#endif /* OXLI_B200_H */
