"""Every k through every hashing and counting route, bit for bit against the CPU oracle, on inputs
built to reach the code that differs per k.

The specialised kernels are one template instance per k of csrc/klist.h: the murmur tail, the
word extraction, the tail mask and the window-validity masks all depend on k.  Every other k runs
the generic kernel.  A wrong hash at one k is silent (the counts still add up; only the keys are
wrong), so random reads are not enough.  The inputs here are built per k with fixed seeds:

1. strand ties: k-mers whose two strands agree on their first t bases and differ at t, for every
   t in 0..k/2, one copy won by each strand (palindromes at t = k/2), also with lower-case bases,
   each placed at every window start residue mod 256 of the batch (the specialised kernels work
   on tiles of 256 window starts, 8 per lane);
2. bad bytes: every byte value 0..255 in clean sequence, and for k > 33 a bad byte at each offset
   33..70 from a lane start at each of the 4 lane offsets of a 32-position mask word;
3. read ends at every residue mod 256, and reads of length k - 1, k, k + 1 and 0;
4. batches with a single bad byte at chosen places (first / last window of the batch or of a
   middle read, inside a read shorter than k, at chosen residues mod 256).
"""
import json
import os
import sys
import threading
from functools import lru_cache

import numpy as np
import pytest

import oracle
from oracle import OracleTable
from oxli_b200._build import specialised_ks

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LISTED = specialised_ks()
GENERIC = [1, 2, 3, 8, 13, 14, 16, 18, 22, 64, 65, 96, 127, 128, 129, 200, 254, 255]
ALL_K = sorted(set(LISTED) | set(GENERIC))
ERROR_RESIDUES = [0, 7, 8, 31, 32, 33, 63, 64, 255]

_COMP = bytes.maketrans(b"ACGTacgt", b"TGCAtgca")
COMP = np.frombuffer(_COMP, dtype=np.uint8)
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
NON_BASES = np.array([v for v in range(256) if v not in b"ACGTacgt"], dtype=np.uint8)


def revcomp(s: bytes) -> bytes:
    return s.translate(_COMP)[::-1]


def shared_prefix(a: bytes, b: bytes) -> int:
    n = 0
    while n < len(a) and a[n] == b[n]:
        n += 1
    return n


def filler(rng, n: int, p_lower: float = 0.1) -> np.ndarray:
    s = ACGT[rng.integers(0, 4, size=n)]
    return s | (rng.random(n) < p_lower).astype(np.uint8) * np.uint8(0x20)


def csr(reads) -> tuple[np.ndarray, np.ndarray]:
    offs = np.zeros(len(reads) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(r) for r in reads])
    bases = np.concatenate(reads).astype(np.uint8) if reads else np.zeros(0, dtype=np.uint8)
    return bases, offs


# ---- input builders ---------------------------------------------------------------------------

@lru_cache(maxsize=None)
def tie_kmers(k: int) -> list[tuple[bytes, int, str]]:
    """(k-mer, t, winner): the forward strand and its reverse complement agree on [0, t) and
    differ at t; winner is 'fw' or 'rc' (the canonical strand) or 'pal' (t = k/2, k even: the
    k-mer is its own reverse complement).  Each k-mer comes once in upper case and once with
    random lower-case bases."""
    rng = np.random.default_rng(1000 + k)
    out = []
    for t in range(k // 2 + 1):
        for fw_wins in (True, False):
            s = ACGT[rng.integers(0, 4, size=k)].copy()
            i = np.arange(t)
            s[k - 1 - i] = COMP[s[i]]
            if 2 * t == k:
                winner = "pal"
            elif 2 * t == k - 1:  # the middle base faces its own complement
                s[t] = rng.choice(np.frombuffer(b"AC" if fw_wins else b"GT", dtype=np.uint8))
                winner = "fw" if fw_wins else "rc"
            else:
                # base t of the forward strand is s[t], of the reverse strand comp(s[k-1-t])
                pairs = [(a, c) for a in b"ACGT" for c in b"ACGT" if a != c and (a < c) == fw_wins]
                a, c = pairs[rng.integers(len(pairs))]
                s[t], s[k - 1 - t] = a, COMP[c]
                winner = "fw" if fw_wins else "rc"
            out.append((s.tobytes(), t, winner))
            low = s | (rng.random(k) < 0.5).astype(np.uint8) * np.uint8(0x20)
            out.append((low.tobytes(), t, winner))
    return out


def tie_batch(k: int):
    """Every tie k-mer at every window start residue mod 256, each in its own short read of
    random filler (the read boundary falls at a random place of the gap between two k-mers).
    Returns (bases, offsets, starts): k-mer m sits at starts[256 m .. 256 m + 255]."""
    rng = np.random.default_rng(2000 + k)
    kmers = np.frombuffer(b"".join(s for s, _, _ in tie_kmers(k)), dtype=np.uint8).reshape(-1, k)
    gap = 3 if (k + 3) % 2 else 4  # odd stride: 256 consecutive placements meet every residue
    stride = k + gap
    n_place = 256 * len(kmers)
    lead = int(rng.integers(0, 256))
    starts = lead + np.arange(n_place, dtype=np.int64) * stride
    stream = filler(rng, lead + n_place * stride)
    span = np.arange(k)
    for m, kmer in enumerate(kmers):
        stream[starts[256 * m:256 * (m + 1), None] + span] = kmer
    cuts = starts[:-1] + k + rng.integers(0, gap + 1, size=n_place - 1)
    empties = cuts[rng.random(len(cuts)) < 0.02]  # a few empty reads
    offs = np.sort(np.concatenate([[0], cuts, empties, [len(stream)]])).astype(np.uint64)
    return stream, offs, starts


def byte_batch(k: int):
    """Every byte value 0..255 four times in clean sequence, bad bytes more than k apart; and
    for k > 33 one bad byte at each offset 33..70 from a lane start, for lane starts at each of
    the offsets 0, 8, 16, 24 of a 32-position mask word.  Returns (bases, offsets, lanes) with
    lanes the (lane start, bad byte position) pairs of the second part."""
    rng = np.random.default_rng(3000 + k)
    values = np.concatenate([rng.permutation(256) for _ in range(4)]).astype(np.uint8)
    pos, at = [], 0
    for i, v in enumerate(values):  # copy q of value v at residue v + 64 q + 17 mod 256
        at += k + 1
        at += (int(v) + 64 * (i // 256) + 17 - at) % 256
        pos.append(at)
    pos = np.array(pos)
    stream = filler(rng, int(pos[-1]) + k + 1)
    stream[pos] = values
    cuts = np.sort(rng.integers(0, len(stream), size=max(len(stream) // (6 * k + 40), 1)))
    reads = np.split(stream, cuts)
    lanes = []
    if k > 33:
        cur = len(stream)
        for sh in (0, 8, 16, 24):
            for d in range(33, 71):
                lane = cur + 64
                lane += (sh + 32 * int(rng.integers(8)) - lane) % 256
                read = filler(rng, lane + d + k + 8 - cur)
                read[lane + d - cur] = rng.choice(NON_BASES)
                reads.append(read)
                lanes.append((lane, lane + d))
                cur += len(read)
    return *csr(reads), lanes


def end_batch(k: int):
    """Reads that end at every residue mod 256, each followed by a read of length k - 1, k,
    k + 1 or 0."""
    rng = np.random.default_rng(4000 + k)
    reads, cur = [], 0
    for i, r in enumerate(rng.permutation(256)):
        n = k + (int(r) - (cur + k)) % 256
        reads.append(filler(rng, n))
        reads.append(filler(rng, max((k - 1, k, k + 1, 0)[i % 4], 0)))
        cur += n + len(reads[-1])
    return csr(reads)


def error_batches(k: int) -> list[tuple[str, np.ndarray, np.ndarray]]:
    """Batches of six clean reads with one bad byte each: in the first / last window of the
    batch, of the middle read (read 3), inside a read shorter than k, and at chosen residues
    mod 256 inside the middle read."""
    rng = np.random.default_rng(5000 + k)
    out = []

    def batch(name, place, short_read=False):
        reads = [filler(rng, k + int(rng.integers(300, 600))) for _ in range(6)]
        if short_read:
            reads.insert(3, filler(rng, k - 1))
        bases, offs = csr(reads)
        p = place(bases, offs)
        bases[p] = NON_BASES[(37 * len(out) + k) % len(NON_BASES)]
        out.append((name, bases, offs))

    batch("first_window", lambda b, o: 0)
    batch("last_window", lambda b, o: len(b) - 1)
    batch("middle_read_first", lambda b, o: int(o[3]))
    batch("middle_read_last", lambda b, o: int(o[4]) - 1)
    if k > 1:
        batch("short_read", lambda b, o: int(o[3]) + (k - 1) // 2, short_read=True)
    for r in ERROR_RESIDUES:
        batch(f"residue_{r}", lambda b, o, r=r: int(o[3]) + (r - int(o[3])) % 256)
    return out


@lru_cache(maxsize=None)
def batches(k: int) -> list[tuple[str, np.ndarray, np.ndarray]]:
    """inputs 1-4 as (name, bases, offsets)"""
    return [("ties", *tie_batch(k)[:2]), ("bytes", *byte_batch(k)[:2]), ("ends", *end_batch(k))] + error_batches(k)


@lru_cache(maxsize=None)
def expected(k: int, i: int, skip: bool):
    """((counted, err_read, err_pos), keys, vals) of batch i in the oracle"""
    _, bases, offs = batches(k)[i]
    ora = OracleTable(k)
    res = ora.consume_batch(bases, offs, skip)
    return res, *ora.items_sorted()


def window_truth(k: int, bases: np.ndarray, offs: np.ndarray) -> np.ndarray:
    """the oracle's per-window hashes of the flat buffer, 0 for windows that straddle two reads"""
    h = oracle.hash_windows(bases, k)
    w = np.arange(len(h), dtype=np.uint64)
    read = np.searchsorted(offs, w, side="right") - 1
    h[w + np.uint64(k) > offs[read + 1]] = 0
    return h


# ---- helpers for the GPU tests ----------------------------------------------------------------

@pytest.fixture(scope="module")
def capi():
    from oxli_b200 import _capi

    assert _capi.lib.oxg_device_count() > 0, "GPU tests need a CUDA device"
    return _capi


def run_ranks(fns):
    """one thread per rank; re-raise the first failure"""
    errs = [None] * len(fns)

    def wrap(i):
        try:
            fns[i]()
        except BaseException as e:  # noqa: BLE001
            errs[i] = e

    ts = [threading.Thread(target=wrap, args=(i,)) for i in range(len(fns))]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=300)
    assert not any(t.is_alive() for t in ts), "a rank hung"
    for e in errs:
        if e is not None:
            raise e


def same_items(got, want) -> bool:
    return len(got[0]) == len(want[0]) and np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


def consume_mismatches(capi, k, pipeline, bases, offs, skip, want, items, label) -> list[str]:
    """one plain-table consume against the oracle's (counted, err_read, err_pos) and table"""
    t = capi.Table(k)
    try:
        got = t.consume_batch(bases, offs, skip)
        status = capi.OK if want[1] < 0 else capi.ERR_BAD_KMER
        errs = []
        if got != (status, *want):
            errs.append(f"{label} {pipeline} skip={skip}: (status, counted, err_read, err_pos) {got} != {(status, *want)}")
        if pipeline == "part" and want[0] > 0 and min(t.last_consume_pass_ms()) <= 0:
            errs.append(f"{label} skip={skip}: the partitioned pipeline did not run")
        if not same_items(t.export(1), items):
            errs.append(f"{label} {pipeline} skip={skip}: table differs from the oracle")
        return errs
    finally:
        t.close()


def shard_mismatches(capi, k, shards, ora, bases, offs, cuts, skip, label) -> list[str]:
    """One collective consume of the reads [cuts[r], cuts[r+1]) on rank r, the same reads into the
    oracle; then the counts, the absorbed windows and the merged shard tables against it."""
    from oxli_b200.sharded import owner_of

    world = len(shards)
    res = [None] * world

    def rank_fn(r):
        def go():
            res[r] = shards[r].consume_batch(bases, offs[cuts[r]:cuts[r + 1] + 1], skip)
        return go

    run_ranks([rank_fn(r) for r in range(world)])
    want, er, ep = ora.consume_batch(bases, offs, skip)
    errs = []
    if sum(x[1] for x in res) != want or sum(x[2] for x in res) != want:
        errs.append(f"{label} skip={skip}: counted {[x[1] for x in res]} absorbed {[x[2] for x in res]}, oracle {want}")
    for r, (st, _, _, r_er, r_ep) in enumerate(res):
        mine = er >= 0 and cuts[r] <= er < cuts[r + 1]
        w = (capi.ERR_BAD_KMER, er - cuts[r], ep) if mine else (capi.OK, -1)
        if (st, r_er, r_ep)[:len(w)] != w:
            errs.append(f"{label} skip={skip}: rank {r} returned {(st, r_er, r_ep)}, expected {w}")
    parts = [s.table.export(1) for s in shards]
    for r, (keys, _) in enumerate(parts):
        if not np.all(owner_of(keys, world) == r):
            errs.append(f"{label} skip={skip}: a key sits on rank {r}, which does not own it")
    allk = np.concatenate([p[0] for p in parts])
    allv = np.concatenate([p[1] for p in parts])
    order = np.argsort(allk, kind="stable")
    if not same_items((allk[order], allv[order]), ora.items_sorted()):
        errs.append(f"{label} skip={skip}: merged shard tables differ from the oracle")
    return errs


def uneven_cuts(n_reads: int, world: int, err_read: int) -> list[int]:
    """Read ranges of the ranks: uneven, and with a bad read on rank 1, every read before it on
    rank 0 and nothing after rank 1 (in error mode the oracle stops at the bad read; a rank that
    held later reads would count them)."""
    if err_read >= 0:
        return [0, err_read // 2] + [n_reads] * (world - 1)
    return [0] + [n_reads * f // (3 * world) for f in range(2, 2 * world, 2)] + [n_reads]


def check_shards(capi, k, world):
    shards = [capi.Shard(k, r, world, device=0, round_windows=1 << 16) for r in range(world)]
    capi.Shard.connect_local(shards)
    ora = OracleTable(k)  # the sharded table accumulates every batch below; so does the oracle
    errs = []
    try:
        for i, (label, bases, offs) in enumerate(batches(k)):
            n = len(offs) - 1
            if i < 3:
                errs += shard_mismatches(capi, k, shards, ora, bases, offs, uneven_cuts(n, world, -1), True, label)
            else:  # single bad byte: skip mode, then error mode with the bad read on rank 1
                errs += shard_mismatches(capi, k, shards, ora, bases, offs, uneven_cuts(n, world, -1), True, label)
                er = expected(k, i, False)[0][1]
                errs += shard_mismatches(capi, k, shards, ora, bases, offs, uneven_cuts(n, world, er), False, label)
    finally:
        for s in shards:
            s.close()
    assert not errs, "\n".join(errs)


# ---- CPU: the builders ------------------------------------------------------------------------

@pytest.mark.parametrize("k", ALL_K)
def test_input_builders(k):
    kmers = tie_kmers(k)
    assert sorted({t for _, t, _ in kmers}) == list(range(k // 2 + 1))
    for s, t, winner in kmers:
        fw = s.upper()
        rc = revcomp(fw)
        assert len(s) == k and set(fw) <= set(b"ACGT")
        if winner == "pal":
            assert 2 * t == k and fw == rc
        else:
            assert shared_prefix(fw, rc) == t, (s, t)
            assert (fw < rc) == (winner == "fw"), (s, t, winner)
        assert oracle.hash_kmer(s) == oracle.hash_kmer(revcomp(s))
    winners = {w for _, _, w in kmers}
    assert winners == ({"fw", "rc", "pal"} if k % 2 == 0 else {"fw", "rc"})

    stream, offs, starts = tie_batch(k)
    assert offs[0] == 0 and offs[-1] == len(stream) and np.all(np.diff(offs.astype(np.int64)) >= 0)
    span = np.arange(k)
    for m, (s, _, _) in enumerate(kmers):  # each copy inside one read, at every residue
        at = starts[256 * m:256 * (m + 1)]
        assert np.all(stream[at[:, None] + span] == np.frombuffer(s, dtype=np.uint8))
        read = np.searchsorted(offs, at.astype(np.uint64), side="right") - 1
        assert np.all(at + k <= offs[read + 1].astype(np.int64))
        assert set((at % 256).tolist()) == set(range(256))

    bases, offs, lanes = byte_batch(k)
    is_bad = np.isin(bases, NON_BASES)
    for v in NON_BASES:  # every non-base value, at several residues
        assert len(set((np.flatnonzero(bases == v) % 256).tolist())) >= 4, v
    bad_at = np.flatnonzero(is_bad)
    assert np.all(np.diff(bad_at) > k)
    if k > 33:
        got = sorted((lane % 32, p - lane) for lane, p in lanes)
        assert got == [(sh, d) for sh in (0, 8, 16, 24) for d in range(33, 71)]
        assert all(is_bad[p] for _, p in lanes)
    else:
        assert lanes == []

    bases, offs = end_batch(k)
    lens = np.diff(offs.astype(np.int64))
    assert set((offs[1:][lens >= k] % 256).tolist()) == set(range(256))
    assert {k - 1, k, k + 1, 0} <= set(lens.tolist())

    for name, bases, offs in error_batches(k):
        bad = np.flatnonzero(np.isin(bases, np.frombuffer(b"acgtACGT", dtype=np.uint8), invert=True))
        assert len(bad) == 1, name
        if name.startswith("residue_"):
            assert bad[0] % 256 == int(name.split("_")[1]) and offs[3] <= bad[0] < offs[4]
    names = [n for n, _, _ in error_batches(k)]
    assert ("short_read" in names) == (k > 1)


# ---- GPU routes -------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("k", ALL_K)
def test_hash_windows(capi, k):
    t = capi.Table(k)
    try:
        for name, bases, _ in batches(k)[:3]:
            got, want = t.hash_windows(bases), oracle.hash_windows(bases, k)
            bad = np.flatnonzero(got != want)
            assert len(bad) == 0, f"{name}: {len(bad)} windows differ, first at {bad[:8]}"
    finally:
        t.close()


@pytest.mark.gpu
@pytest.mark.parametrize("k", ALL_K)
def test_hash_batch_device(capi, k):
    t = capi.Table(k)
    try:
        for i, (name, bases, offs) in enumerate(batches(k)[:3]):
            n_win = len(bases) - k + 1
            got = np.zeros(n_win, dtype=np.uint64)
            d_b, d_o = capi.device_alloc(len(bases) + 64), capi.device_alloc(offs.nbytes)
            d_h = capi.device_alloc(n_win * 8)
            try:
                capi.h2d(d_b, bases); capi.h2d(d_o, offs)
                t.hash_batch_device(d_b, d_o, len(offs) - 1, len(bases), d_h)
                capi.d2h(got, d_h)
                t.clear()
                counted = t.count_hashes_device(d_h, n_win, skip_zero=True)
            finally:
                capi.device_free(d_b); capi.device_free(d_o); capi.device_free(d_h)
            bad = np.flatnonzero(got != window_truth(k, bases, offs))
            assert len(bad) == 0, f"{name}: {len(bad)} windows differ, first at {bad[:8]}"
            (want, _, _), keys, vals = expected(k, i, True)
            assert counted == want, name
            assert same_items(t.export(1), (keys, vals)), name
    finally:
        t.close()


@pytest.mark.gpu
@pytest.mark.parametrize("k", ALL_K)
def test_consume_fused(capi, k):
    capi.set_pipeline("fused")
    try:
        errs = []
        for i, (name, bases, offs) in enumerate(batches(k)):
            for skip in (True, False):
                want, keys, vals = expected(k, i, skip)
                errs += consume_mismatches(capi, k, "fused", bases, offs, skip, want, (keys, vals), name)
    finally:
        capi.set_pipeline("auto")
    assert not errs, "\n".join(errs)


@pytest.mark.gpu
@pytest.mark.parametrize("k", LISTED)
def test_consume_part(capi, k):
    capi.set_pipeline("part")
    try:
        errs = []
        for i, (name, bases, offs) in enumerate(batches(k)):
            for skip in (True, False):
                want, keys, vals = expected(k, i, skip)
                errs += consume_mismatches(capi, k, "part", bases, offs, skip, want, (keys, vals), name)
    finally:
        capi.set_pipeline("auto")
    assert not errs, "\n".join(errs)


@pytest.mark.gpu
@pytest.mark.parametrize("k", LISTED)
def test_shard_world2(capi, k):
    check_shards(capi, k, 2)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [15, 33, 63])
def test_shard_world4(capi, k):
    check_shards(capi, k, 4)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [15, 33, 63, 64, 255])
def test_hash_windows_piece_seam(capi, k):
    """one sequence of 4 Mi + 300 windows: the host copies and hashes it in pieces of 4 Mi"""
    seam = 4 << 20
    rng = np.random.default_rng(6000 + k)
    seq = filler(rng, seam + 300 + k - 1)
    for p in (seam - 1, seam + k - 2, seam + k + 5, seam - k - 3):
        seq[p] = rng.choice(NON_BASES)
    t = capi.Table(k)
    try:
        got = t.hash_windows(seq)
    finally:
        t.close()
    want = oracle.hash_windows(seq, k)
    assert len(got) == seam + 300
    bad = np.flatnonzero(got != want)
    assert len(bad) == 0, f"{len(bad)} windows differ, first at {bad[:8]}"
    assert np.count_nonzero(want[seam - k:seam + k] == 0) > 0  # the bad bytes sit across the seam


# ---- a host batch streamed in 1 MiB chunks ----------------------------------------------------

CHUNK_TOTAL = 6 << 20


@lru_cache(maxsize=1)
def _chunk_source() -> np.ndarray:
    from oracle.synth import synth_reads

    return synth_reads(CHUNK_TOTAL // 150 + 1, 150, 200_000, seed=8, sub_ppm=2000)[:CHUNK_TOTAL]


def chunked_batch(k: int):
    """About 6 MB of reads of 0..300 bases.  At the 1 MiB seams 1 and 2 a short read straddles
    the seam between two long ones; at the seams 3, 4 and 5 MiB one read of at least 4k bases
    holds two bad bytes within k of the seam."""
    rng = np.random.default_rng(7000 + k)
    bases = _chunk_source().copy()
    ends = np.cumsum(rng.integers(0, 301, size=CHUNK_TOTAL // 100))
    ends = ends[ends < CHUNK_TOTAL]
    seams = np.arange(1, 6, dtype=np.int64) << 20
    for s in seams:
        ends = ends[np.abs(ends - s) > 2 * k + 600]
    near = np.where(seams < 3 << 20, 1, 2 * k)
    cuts = [ends, seams - near - rng.integers(0, k, 5), seams + near + rng.integers(0, 3, 5)]
    offs = np.sort(np.concatenate([[0], *cuts, [CHUNK_TOTAL]])).astype(np.uint64)
    for s in seams[2:]:
        bases[s - 1 - rng.integers(0, k)] = ord("N")
        bases[s + rng.integers(0, k)] = rng.choice(NON_BASES)
    return bases, offs


def _chunked_worker(ks, out_path):
    """Runs in a spawned process whose OXLI_B200_CHUNK_MB is 1: the library reads it once, when
    it loads.  Writes {k: [mismatch, ...]} to out_path."""
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oxli_b200 import _capi as capi

    results = {}
    for k in ks:
        bases, offs = chunked_batch(k)
        errs = []
        truth = {}
        for skip in (True, False):
            ora = OracleTable(k)
            truth[skip] = (ora.consume_batch(bases, offs, skip, nthreads=4), ora.items_sorted())
        if truth[False][0][1] < 0:
            errs.append("the batch has no bad window in error mode")
        for pipeline in ("fused", "part") if k in LISTED else ("fused",):
            capi.set_pipeline(pipeline)
            for skip in (True, False):
                want, items = truth[skip]
                errs += consume_mismatches(capi, k, pipeline, bases, offs, skip, want, items, "chunked")
        capi.set_pipeline("auto")
        if k in LISTED:
            shards = [capi.Shard(k, r, 2, device=0, round_windows=1 << 16) for r in range(2)]
            capi.Shard.connect_local(shards)
            ora = OracleTable(k)
            n = len(offs) - 1
            errs += shard_mismatches(capi, k, shards, ora, bases, offs, uneven_cuts(n, 2, -1), True, "chunked")
            for s in shards:
                s.close()
            shards = [capi.Shard(k, r, 2, device=0, round_windows=1 << 16) for r in range(2)]
            capi.Shard.connect_local(shards)
            ora = OracleTable(k)
            cuts = uneven_cuts(n, 2, truth[False][0][1])
            errs += shard_mismatches(capi, k, shards, ora, bases, offs, cuts, False, "chunked")
            for s in shards:
                s.close()
        results[k] = errs
    with open(out_path, "w") as f:
        json.dump(results, f)


@pytest.fixture(scope="module")
def chunked_results(capi, tmp_path_factory):
    import multiprocessing as mp

    out = str(tmp_path_factory.mktemp("chunked") / "results.json")
    old = os.environ.get("OXLI_B200_CHUNK_MB")
    os.environ["OXLI_B200_CHUNK_MB"] = "1"
    try:
        p = mp.get_context("spawn").Process(target=_chunked_worker, args=(ALL_K, out))
        p.start()
    finally:
        if old is None:
            del os.environ["OXLI_B200_CHUNK_MB"]
        else:
            os.environ["OXLI_B200_CHUNK_MB"] = old
    p.join(timeout=1800)
    if p.is_alive():
        p.kill()
        p.join()
    assert p.exitcode == 0, f"the chunked-batch process exited with {p.exitcode}"
    with open(out) as f:
        return {int(k): v for k, v in json.load(f).items()}


@pytest.mark.gpu
@pytest.mark.parametrize("k", ALL_K)
def test_host_batch_in_1mib_chunks(chunked_results, k):
    assert chunked_results[k] == []


# ---- refusals ---------------------------------------------------------------------------------

@pytest.mark.gpu
def test_refusals(capi):
    for k in (0, 256):
        with pytest.raises(capi.OxliError) as e:
            capi.Table(k)
        assert e.value.status == capi.ERR_INVALID
    for k in GENERIC:
        with pytest.raises(capi.OxliError) as e:
            capi.Shard(k, 0, 1)
        assert e.value.status == capi.ERR_INVALID and "klist.h" in str(e.value), k
