"""Point lookups on the hash-sharded table (oxg_shard_get_hashes*, ShardedTable.get*) against the
unsharded oracle.

Every rank asks for its own list of hashes; each hash is answered by the rank that owns it, in
exchange rounds of the same kind as a consume call's.  The lists mix present keys of every owner,
absent keys, 0, 2^64-1 (kept in its owner's side entry) and duplicates, differ in size between
ranks (one rank asks nothing) and are longer than one round carries.  As in test_gpu_sharded.py,
several shards on one GPU run the same code as one shard per GPU."""
import os
import sys
import threading
import time

import numpy as np
import pytest

from oracle import OracleTable
from synth import synth_reads, uniform_offsets

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOP = (1 << 64) - 1


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


def devices_for(capi, world):
    n = capi.lib.oxg_device_count()
    return [r % n for r in range(world)]


def expected(q, tk, tv, side=None):
    """the oracle's answer to every query (0 when absent); side = value set for 2^64-1"""
    q = np.asarray(q, dtype=np.uint64)
    i = np.minimum(np.searchsorted(tk, q), len(tk) - 1)
    out = np.where(tk[i] == q, tv[i], 0).astype(np.uint64)
    if side is not None:
        out[q == np.uint64(TOP)] = side
    return out


def make_queries(rng, tk, size):
    """half present keys (drawn with replacement: duplicates), half random u64 (absent), plus 0,
    2^64-1 and repeats, shuffled"""
    if size == 0:
        return np.zeros(0, dtype=np.uint64)
    n_present = size // 2 - 8
    present = tk[rng.integers(0, len(tk), n_present)]
    absent = rng.integers(0, TOP, size - n_present - 8, dtype=np.uint64, endpoint=True)
    extra = np.concatenate([np.array([0, TOP, 0, TOP], dtype=np.uint64), present[:4]])
    q = np.concatenate([present, absent, extra])
    rng.shuffle(q)
    return q


def consumed_shards(capi, world, k, bases, offs, round_windows=1 << 16):
    from oxli_b200.sharded import ShardedTable, split_reads

    shards = ShardedTable.local(k, world, devices_for(capi, world), round_windows=round_windows)
    n = len(offs) - 1

    def consume(r):
        lo, hi = split_reads(n, r, world)
        shards[r].consume_batch(bases, offs[lo:hi + 1])

    run_ranks([lambda r=r: consume(r) for r in range(world)])
    return shards


def lookup_all(shards, queries):
    got = [None] * len(shards)

    def go(r):
        got[r] = shards[r].get_hash_array(queries[r])

    run_ranks([lambda r=r: go(r) for r in range(len(shards))])
    return got


# "staged": rounds of 2.5 Mi queries, so that a host list's round crosses in several pieces of the
# shard's 1 Mi-entry staging buffer (on ranks 0 and 2), the last of them partly filled
@pytest.mark.parametrize("world,round_windows", [(1, 1 << 16), (2, 1 << 16), (4, 1 << 16), (8, 1 << 16), (4, 5 << 19)],
                         ids=["1", "2", "4", "8", "4-staged"])
def test_lookups_in_one_process_vs_oracle(capi, world, round_windows):
    from oxli_b200.sharded import owner_of

    k = 21 if world % 4 else 31
    n, L, G = 24_000, 150, 150_000
    bases = synth_reads(n, L, G, seed=71, sub_ppm=5000, n_ppm=800)
    offs = uniform_offsets(n, L)
    truth = OracleTable(k)
    truth.consume_batch(bases, offs, True, nthreads=4)
    tk, tv = truth.items_sorted()
    shards = consumed_shards(capi, world, k, bases, offs, round_windows)
    Q = shards[0].engine.info()["round_windows"]  # queries per rank and round
    assert Q >= round_windows
    # rank 0 needs three rounds; the others ask less, and rank 1 nothing at all
    sizes = [2 * Q + 1] + [0 if r == 1 else Q // r + r for r in range(1, world)]
    rng = np.random.default_rng(world)
    queries = [make_queries(rng, tk, s) for s in sizes]
    assert set(owner_of(queries[0], world).tolist()) == set(range(world))

    got = lookup_all(shards, queries)
    for q, a in zip(queries, got):
        assert a.dtype == np.uint64 and len(a) == len(q)
        assert np.array_equal(a, expected(q, tk, tv))
    # 2^64-1 enters its owner's side entry: present with count 0 (answers 0), then with 7
    owner = world - 1
    for value in (0, 7):
        shards[owner].engine.table.set_hash(TOP, value)
        got = lookup_all(shards, queries)
        for q, a in zip(queries, got):
            assert np.array_equal(a, expected(q, tk, tv, side=value))

    # single k-mers and hashes, every rank its own
    text = bases.tobytes().decode()
    kmers = []
    for r in range(world):  # the first k-mer of read r without an N (every rank must take part)
        at = r * L
        while "N" in text[at:at + k]:
            at += 1
        kmers.append(text[at:at + k])
    single = [None] * world

    def one(r):
        single[r] = (shards[r].get(kmers[r]), shards[r].get_hash(TOP), shards[r].get_hash(int(tk[r])))

    run_ranks([lambda r=r: one(r) for r in range(world)])
    for r in range(world):
        assert single[r] == (truth.get(kmers[r]), 7, int(tv[r])) and single[r][0] > 0
    with pytest.raises(ValueError, match="kmer size does not match count table ksize"):
        shards[0].get("ACGT")  # refused before the lookup: no rank is left waiting
    for s in shards:
        s.close()


def test_lookups_between_consume_calls(capi):
    """consume, look up, consume the same reads again, look up: every answer doubles (consume and
    lookup rounds share the round count and the parity of the exchange buffers)"""
    from oxli_b200.sharded import split_reads

    world, k = 2, 31
    n, L, G = 16_000, 150, 100_000
    bases = synth_reads(n, L, G, seed=5, sub_ppm=3000, n_ppm=500)
    offs = uniform_offsets(n, L)
    truth = OracleTable(k)
    truth.consume_batch(bases, offs, True, nthreads=4)
    tk, tv = truth.items_sorted()
    shards = consumed_shards(capi, world, k, bases, offs)
    Q = shards[0].engine.info()["round_windows"]
    rng = np.random.default_rng(11)
    queries = [make_queries(rng, tk, Q + 5), make_queries(rng, tk, Q // 2)]
    first = lookup_all(shards, queries)

    def again(r):
        lo, hi = split_reads(n, r, world)
        shards[r].consume_batch(bases, offs[lo:hi + 1])

    run_ranks([lambda r=r: again(r) for r in range(world)])
    second = lookup_all(shards, queries)
    for q, a, b in zip(queries, first, second):
        assert np.array_equal(a, expected(q, tk, tv))
        assert np.array_equal(b, 2 * a)
    for s in shards:
        s.close()


def test_lookups_from_device_lists(capi):
    world, k = 2, 21
    n, L, G = 16_000, 150, 100_000
    bases = synth_reads(n, L, G, seed=19, sub_ppm=5000, n_ppm=800)
    offs = uniform_offsets(n, L)
    truth = OracleTable(k)
    truth.consume_batch(bases, offs, True, nthreads=4)
    tk, tv = truth.items_sorted()
    shards = consumed_shards(capi, world, k, bases, offs)
    devs = devices_for(capi, world)
    Q = shards[0].engine.info()["round_windows"]
    rng = np.random.default_rng(3)
    queries = [make_queries(rng, tk, 2 * Q + 9), make_queries(rng, tk, Q // 3)]
    # device buffers are made before the ranks start (cudaMalloc / cudaFree synchronise the device,
    # and a rank must not wait for the device while a peer on it waits for that rank)
    bufs = []
    for r in range(world):
        d_q = capi.device_alloc(len(queries[r]) * 8, devs[r]); d_out = capi.device_alloc(len(queries[r]) * 8, devs[r])
        capi.h2d(d_q, queries[r], devs[r])
        bufs.append((d_q, d_out))

    def go(r):
        shards[r].engine.get_hashes_device(bufs[r][0], len(queries[r]), bufs[r][1])

    run_ranks([lambda r=r: go(r) for r in range(world)])
    for r, (d_q, d_out) in enumerate(bufs):
        got = np.zeros(len(queries[r]), dtype=np.uint64)
        capi.d2h(got, d_out, devs[r])
        back = np.zeros(len(queries[r]), dtype=np.uint64)
        capi.d2h(back, d_q, devs[r])
        capi.device_free(d_q, devs[r]); capi.device_free(d_out, devs[r])
        assert np.array_equal(got, expected(queries[r], tk, tv))
        assert np.array_equal(back, queries[r])  # the query list itself is left as it was
    for s in shards:
        s.close()


def _lookup_worker(rank, world, k, conns, out_dir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oxli_b200 import _capi as capi
    from oxli_b200.sharded import ShardedTable, split_reads
    from synth import synth_reads, uniform_offsets

    def exchange(blob):
        # star all-gather over pipes: rank 0 collects and hands the list back
        if rank == 0:
            got = [blob] + [c.recv() for c in conns]
            for c in conns:
                c.send(got)
            return got
        conns.send(blob)
        return conns.recv()

    dev = rank % capi.lib.oxg_device_count()
    n, L, G = 20_000, 150, 120_000
    bases = synth_reads(n, L, G, seed=13, n_ppm=500)
    offs = uniform_offsets(n, L)
    t = ShardedTable(k, rank, world, device=dev, exchange=exchange, round_windows=1 << 16)
    lo, hi = split_reads(n, rank, world)
    t.consume_batch(bases, offs[lo:hi + 1])
    Q = t.engine.info()["round_windows"]
    rng = np.random.default_rng(40 + rank)
    # the windows of 2000 reads (present keys of both owners; 0 for windows across an N) and
    # random absent keys: two rounds on rank 0, one on rank 1
    present = t.engine.table.hash_windows(bases[rank * 2000 * L:(rank + 1) * 2000 * L])
    absent = rng.integers(0, TOP, (Q + 1000) if rank == 0 else Q // 4, dtype=np.uint64, endpoint=True)
    q = np.concatenate([present, absent, np.array([0, TOP], dtype=np.uint64), present[:100]])
    rng.shuffle(q)
    answers = t.get_hash_array(q)
    np.savez(os.path.join(out_dir, f"lookup{rank}.npz"), queries=q, answers=answers)
    exchange(b"done")  # nobody unmaps an exchange area a peer may still be reading or answering into
    t.close()


def test_lookups_in_separate_processes_over_cuda_ipc(capi, tmp_path):
    import multiprocessing as mp

    world, k = 2, 31
    ctx = mp.get_context("spawn")
    a, b = ctx.Pipe()
    procs = [ctx.Process(target=_lookup_worker, args=(0, world, k, [a], str(tmp_path))),
             ctx.Process(target=_lookup_worker, args=(1, world, k, b, str(tmp_path)))]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    n, L, G = 20_000, 150, 120_000
    truth = OracleTable(k)
    truth.consume_batch(synth_reads(n, L, G, seed=13, n_ppm=500), uniform_offsets(n, L), True, nthreads=4)
    tk, tv = truth.items_sorted()
    for r in range(world):
        part = np.load(tmp_path / f"lookup{r}.npz")
        want = expected(part["queries"], tk, tv)
        assert np.count_nonzero(want) > 100_000
        assert np.array_equal(part["answers"], want)


def test_refused_calls_start_no_exchange(capi):
    from oxli_b200.sharded import ShardedTable

    err_invalid = capi.ERR_INVALID
    lib = capi.lib
    h = np.array([5, 9, 7, TOP], dtype=np.uint64)
    out = np.zeros(4, dtype=np.uint64)
    s = capi.Shard(21, 0, 1)
    assert lib.oxg_shard_get_hashes(s._h, None, 4, out.ctypes.data) == err_invalid
    assert lib.oxg_shard_get_hashes(s._h, h.ctypes.data, 4, None) == err_invalid
    d = capi.device_alloc(32)
    assert lib.oxg_shard_get_hashes_device(s._h, None, 4, d) == err_invalid
    assert lib.oxg_shard_get_hashes_device(s._h, h.ctypes.data, 4, d) == err_invalid  # a host list
    capi.device_free(d)
    s.table.count_hashes([5, 5, 9])
    assert s.get_hashes(h).tolist() == [2, 1, 0, 0]
    assert s.get_hashes(h[:0]).tolist() == []
    s.close()
    # a shard whose peers are not connected: refused at once
    lone = capi.Shard(21, 0, 2)
    assert lib.oxg_shard_get_hashes(lone._h, h.ctypes.data, 4, out.ctypes.data) == err_invalid
    assert b"not connected" in lib.oxg_last_error()
    lone.close()
    # a refused call on one rank of a connected pair returns at once: had it started an exchange,
    # it would have waited for the other rank; both ranks then look up together as usual
    pair = ShardedTable.local(21, 2, devices_for(capi, 2))
    t0 = time.monotonic()
    assert lib.oxg_shard_get_hashes(pair[0].engine._h, None, 4, out.ctypes.data) == err_invalid
    assert time.monotonic() - t0 < 5
    pair[0].engine.table.count_hashes([5, 5, 9])
    pair[1].engine.table.set_hash(TOP, 3)
    got = lookup_all(pair, [h, np.array([TOP, 5], dtype=np.uint64)])
    assert got[0].tolist() == [2, 1, 0, 3] and got[1].tolist() == [3, 2]
    for p in pair:
        p.close()
