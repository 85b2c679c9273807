"""Hash-sharded k-mer count table across the GPUs of one node: the Python face of the
`oxg_shard_*` entry points (include/oxli_b200.h).

The table is sharded by the high bits of the hash -- owner(h) = h >> (64 - log2 N) -- as
BASELINE.json's north_star prescribes; every rank hashes its own reads, leaves the hashes in
fragments per (owner, table partition) in its own HBM, and each owner's aggregation kernel
pulls its fragments from all ranks over NVLink (peer-mapped memory) and counts them.  Point
queries (get / get_hash / get_hash_array, src/lib.rs:170-194) take the same route: every rank
sends its hashes to their owners, which answer them in place.  So does `add` (KmerCountTable::add,
src/lib.rs:778-837) of a table counted on one GPU: every (key, count) of each rank's plain table
goes to its owner and is added there; a second sharded table is added rank by rank, its shards
already on their owners.  Removal takes the same route: drop / drop_hash / drop_hash_array
(src/lib.rs:197-224) send each hash to its owner, which erases it, and mincut / maxcut
(src/lib.rs:227-267) cut every shard and sum what each removed.  export and dump (src/lib.rs:330-381)
need no routing at all: every key of rank r is below every key of rank r + 1, so each rank sorts
and formats its own shard and writes its part of one file.  Neither do union, intersection,
difference, symmetric_difference and cosine of two tables sharded the same way (src/lib.rs:610-655,
727-765): a key of rank r can only meet keys of rank r, so each rank computes its own part.  All of that, including the
rank-to-rank flags and the reductions (len / sum / min / max, histo, |A & B|, jaccard, digests:
reference src/lib.rs:464-539, 610-638, 708-722), lives in the C library.

Nothing here imports torch.  A launcher (bench.py, the tests, a user's torchrun script)
provides ONE thing: `exchange(blob: bytes) -> list[bytes]`, an all-gather of a 64-byte CUDA IPC
handle among the ranks at construction time -- any transport will do (torch.distributed,
MPI, a pipe).  Ranks that live in one process use `ShardedTable.local(...)` instead.

The per-rank engine is injectable, so the host-side logic in this file (owner function, the
split of a read set among ranks, zero-filled histograms, error mapping) is testable on CPU
with world_size 2 over gloo; the product engine is `_capi.Shard`.
"""
from __future__ import annotations

import numpy as np


def owner_of(h: np.ndarray | int, world: int):
    """Shard that owns hash h: the top log2(world) bits."""
    if world == 1:
        return h * 0 if isinstance(h, np.ndarray) else 0
    shift = 64 - (world.bit_length() - 1)
    if isinstance(h, np.ndarray):
        return (np.asarray(h, dtype=np.uint64) >> np.uint64(shift)).astype(np.int64)
    return int(h) >> shift


def split_reads(n_reads: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous block of a read set that rank `rank` ingests (any split works: counts add)."""
    return n_reads * rank // world, n_reads * (rank + 1) // world


class BadKmerError(ValueError):
    """consume met a non-ACGT window in error mode (reference: src/lib.rs:593-596)."""

    def __init__(self, position: int, read: int):
        super().__init__(f"bad k-mer encountered at position {position}")
        self.position, self.read = position, read


_ERR_INVALID, _ERR_NOMEM = 2, 4  # oxg_status (include/oxli_b200.h)


def _engine_call(fn, *args):
    """fn(*args), with the engine's refusals raised as ValueError and its failed device reservations
    as MemoryError (the engine's error stays chained)"""
    try:
        return fn(*args)
    except RuntimeError as e:
        status = getattr(e, "status", None)
        if status == _ERR_INVALID:
            raise ValueError(str(e)) from e
        if status == _ERR_NOMEM:
            raise MemoryError(str(e)) from e
        raise


class ShardedTable:
    """Rank-local handle on a hash-sharded count table.  Methods marked (collective) must be
    called by every rank."""

    def __init__(self, ksize: int, rank: int, world: int, device: int = 0, exchange=None,
                 capacity_hint: int = 0, round_windows: int = 0, engine=None):
        assert world >= 1 and world & (world - 1) == 0, "number of shards must be a power of two"
        self.ksize, self.rank, self.world = ksize, rank, world
        if engine is None:
            from . import _capi as capi  # fails loudly without the CUDA library: there is no CPU engine in the product

            engine = capi.Shard(ksize, rank, world, device=device, capacity_hint=capacity_hint, round_windows=round_windows)
        self.engine = engine
        if world > 1 and exchange is not None:
            handles = exchange(engine.export_handle())
            assert len(handles) == world
            engine.connect(list(handles))

    @classmethod
    def local(cls, ksize: int, world: int, devices: list[int], capacity_hint: int = 0, round_windows: int = 0):
        """All shards in this process (one driver over a node's GPUs, or N > 1 on one GPU in tests).
        Collective calls must then be issued from one thread per shard."""
        from . import _capi as capi

        shards = [cls(ksize, r, world, device=devices[r % len(devices)], capacity_hint=capacity_hint,
                      round_windows=round_windows) for r in range(world)]
        capi.Shard.connect_local([s.engine for s in shards])
        return shards

    def close(self):
        self.engine.close()

    # -- ingest (collective) ----------------------------------------------------------
    def consume_batch(self, bases: np.ndarray, offsets: np.ndarray, skip_bad_kmers: bool = True) -> int:
        """This rank's reads (CSR batch in host memory).  Returns the number of k-mers counted
        from them, i.e. the sum of what the reference's consume would return per read."""
        st, counted, absorbed, er, ep = self.engine.consume_batch(bases, offsets, skip_bad_kmers)
        self.last_absorbed = absorbed
        if st != 0:
            raise BadKmerError(ep, er)
        return counted

    def consume_batch_device(self, d_bases: int, d_offsets: int, n_reads: int, total_bases: int,
                             skip_bad_kmers: bool = True) -> int:
        st, counted, absorbed, er, ep = self.engine.consume_batch_device(d_bases, d_offsets, n_reads, total_bases, skip_bad_kmers)
        self.last_absorbed = absorbed
        if st != 0:
            raise BadKmerError(ep, er)
        return counted

    # -- lookups (collective) ----------------------------------------------------------
    def get_hash_array(self, hashes) -> np.ndarray:
        """Counts of this rank's hashes in the whole table (0 when absent), in order
        (src/lib.rs:185-194).  Every rank calls it with its own list, empty ones included; each
        hash is answered by the rank that owns it."""
        return self.engine.get_hashes(hashes)

    def get_hash(self, h: int) -> int:
        return int(self.get_hash_array([h])[0])

    def _hash_kmer(self, kmer: str) -> int:
        """The k-mer's hash, through this rank's shard table.  A k-mer of the wrong length or with
        a non-ACGT base raises here, before the caller starts an exchange; the other ranks' call
        then fails once the exchange gives up waiting for this one."""
        if len(kmer) != self.ksize:
            raise ValueError("kmer size does not match count table ksize")
        h = self.engine.table.hash_windows(kmer.encode())
        if h[0] == 0:  # (the reference panics here; the drop-in raises the same error)
            raise RuntimeError(f"invalid DNA character in input k-mer: {kmer}")
        return int(h[0])

    def get(self, kmer: str) -> int:
        """Count of a k-mer (src/lib.rs:170-182)."""
        return self.get_hash(self._hash_kmer(kmer))

    # -- merges (collective) -----------------------------------------------------------
    def add(self, other) -> tuple[int, int]:
        """KmerCountTable::add (src/lib.rs:778-837): counts[h] += other[h] for every key of
        `other`.  Every rank calls it: with another ShardedTable (same world, rank by rank; each
        rank adds that table's shard into its own), or each with its own plain `_capi.Table` on
        this rank's device, or None to add nothing (each key of a plain table is sent to the rank
        that owns it).  `other` is not modified.  Returns (counts_added, new_keys) over the whole
        table, the two numbers the reference prints; this class prints nothing (the drop-in
        KmerCountTable does)."""
        if other is self or other is self.engine.table:
            raise ValueError("cannot add a table to itself")
        if other is not None and other.ksize != self.ksize:
            raise ValueError("KmerCountTables must have the same ksize")
        if isinstance(other, ShardedTable):
            return self.engine.merge(other.engine)
        return self.engine.merge_table(other)

    # -- removal (collective) ---------------------------------------------------------
    def drop_hash_array(self, hashes) -> int:
        """drop_hash (src/lib.rs:213-224) for each of this rank's hashes on the whole table: every
        rank calls it with its own list, empty ones included, and each hash is removed by the rank
        that owns it.  Returns the distinct keys removed from the whole table."""
        return self.engine.erase_hashes(hashes)

    def drop_hash(self, h: int) -> None:
        self.drop_hash_array([h])

    def drop(self, kmer: str) -> None:
        """drop (src/lib.rs:197-224)."""
        self.drop_hash(self._hash_kmer(kmer))

    def mincut(self, m: int) -> int:
        """Removes every key with a count below m from every shard (src/lib.rs:227-267); returns
        the keys removed from the whole table."""
        return self.engine.cut(0, m)

    def maxcut(self, m: int) -> int:
        """Removes every key with a count above m from every shard (src/lib.rs:227-267); returns the
        keys removed from the whole table."""
        return self.engine.cut(1, m)

    # -- reductions (collective) ------------------------------------------------------
    def stats(self) -> dict:
        return self.engine.stats()

    def __len__(self) -> int:
        return self.stats()["len"]

    def histo(self, zero: bool = True) -> list[tuple[int, int]]:
        sparse = self.engine.histo()
        if not zero:
            return sparse
        merged = dict(sparse)
        top = sparse[-1][0] if sparse else 0
        return [(f, merged.get(f, 0)) for f in range(top + 1)]  # src/lib.rs:475-480

    def setop_sizes(self, other: "ShardedTable") -> tuple[int, int]:
        return self.engine.setop_sizes(other.engine)

    def jaccard(self, other: "ShardedTable") -> float:
        return self.engine.jaccard(other.engine)

    # -- set operations and cosine (collective) ------------------------------------------
    def _setop(self, other: "ShardedTable", op: int) -> tuple[np.ndarray, int, int]:
        if not isinstance(other, ShardedTable):
            raise TypeError(f"expected a ShardedTable, got {type(other).__name__}")
        return _engine_call(self.engine.setop, other.engine, op)

    def union(self, other: "ShardedTable") -> tuple[np.ndarray, int, int]:
        """union (src/lib.rs:610-655) with a table sharded the same way.  Returns (keys, start, total):
        the keys of the result that this rank owns in ascending order, their position in the whole
        sorted result and its size.  A key of A owned by rank r can only be in B's shard on rank r,
        so each rank computes its part on its GPU and no key crosses between GPUs; the parts in rank
        order are the whole result sorted.  A key held with count 0 is a member."""
        return self._setop(other, 0)

    def intersection(self, other: "ShardedTable") -> tuple[np.ndarray, int, int]:
        """intersection (src/lib.rs:610-655); returns this rank's (keys, start, total) as union."""
        return self._setop(other, 1)

    def difference(self, other: "ShardedTable") -> tuple[np.ndarray, int, int]:
        """difference (src/lib.rs:610-655); returns this rank's (keys, start, total) as union."""
        return self._setop(other, 2)

    def symmetric_difference(self, other: "ShardedTable") -> tuple[np.ndarray, int, int]:
        """symmetric_difference (src/lib.rs:610-655); returns this rank's (keys, start, total) as union."""
        return self._setop(other, 3)

    def cosine(self, other: "ShardedTable") -> float:
        """cosine similarity of the count vectors (src/lib.rs:727-765) with a table sharded the same
        way: the same float on every rank; 0.0 when either whole table is empty or a norm is 0."""
        if not isinstance(other, ShardedTable):
            raise TypeError(f"expected a ShardedTable, got {type(other).__name__}")
        return _engine_call(self.engine.cosine, other.engine)

    def digest(self) -> dict:
        """{n, sum, xor, sum_hc, foreign} of the whole table; foreign must be 0."""
        return self.engine.digest()

    # -- export and dump (collective) ---------------------------------------------------
    @staticmethod
    def _sort_mode(sortcounts: bool, sortkeys: bool) -> int:
        if sortcounts and sortkeys:
            raise ValueError("Cannot sort by both counts and keys at the same time.")
        return 1 if sortkeys else 2 if sortcounts else 0

    def export(self, sortcounts: bool = False, sortkeys: bool = False):
        """This rank's part of the whole table in dump order (src/lib.rs:330-381): by key with
        sortkeys, by (count, key) with sortcounts, else each rank's shard in table order.  Returns
        (keys, vals, runs, total): this rank's pairs, an (n_runs, 2) array of (global_start, length)
        pieces that place keys / vals in the whole table in order, and the whole table's length.
        Every key of rank r is below every key of rank r + 1, so each rank sorts its own shard on
        its GPU and no pair crosses between GPUs."""
        return self.engine.export_pairs(self._sort_mode(sortcounts, sortkeys))

    def dump(self, file: str, sortcounts: bool = False, sortkeys: bool = False) -> None:
        """dump(file, sortcounts, sortkeys) of the whole table (src/lib.rs:330-381): every rank
        passes the same path, and the ranks write one file of "<hash>\\t<count>\\n" lines together.
        With sortkeys or sortcounts it holds the bytes the drop-in KmerCountTable.dump writes for a
        table of the same pairs; without, the same lines, each rank's shard in one block, the blocks
        in rank order.  A file that cannot be written raises OSError on every rank."""
        self.engine.dump(file, self._sort_mode(sortcounts, sortkeys))

    # -- this rank's shard only ---------------------------------------------------------
    def local_items_sorted(self):
        return self.engine.table.export(1)
