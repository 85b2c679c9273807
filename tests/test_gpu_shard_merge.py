"""Adding tables into the hash-sharded table (oxg_shard_merge_table / oxg_shard_merge,
ShardedTable.add) against a host model of KmerCountTable::add (src/lib.rs:778-837).

Every rank adds its own plain table: each (key, count) travels to the rank that owns the key in
exchange rounds of the same kind as consume and lookup rounds, and is added there.  A second
sharded table is added rank by rank.  As in test_gpu_shard_lookup.py, several shards on one GPU
run the same code as one shard per GPU."""
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
M64 = 1 << 64
L, G = 150, 150_000


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


def each_rank(shards, fn):
    """fn(r) on every rank at once (collective calls); returns the results in rank order"""
    out = [None] * len(shards)

    def go(r):
        out[r] = fn(r)

    run_ranks([lambda r=r: go(r) for r in range(len(shards))])
    return out


def reads(seed, n, first_read=0):
    """n reads of the genome of `seed` (the same genome for every first_read: reads overlap)"""
    return synth_reads(n, L, G, seed=seed, first_read=first_read, sub_ppm=5000, n_ppm=800), uniform_offsets(n, L)


def oracle_dict(k, bases, offs):
    t = OracleTable(k)
    t.consume_batch(bases, offs, True, nthreads=4)
    tk, tv = t.items_sorted()
    return dict(zip(tk.tolist(), tv.tolist()))


def model_add(d, keys, vals):
    """KmerCountTable::add of (keys, vals) into dict d, in order: (counts added, new keys)"""
    added = fresh = 0
    for h, v in zip(keys.tolist(), vals.tolist()):
        before = d.get(h, 0)
        fresh += before == 0
        d[h] = (before + v) % M64
        added += v
    return added % M64, fresh


def check_against(shards, d, world):
    """every rank holds exactly its owners' slice of d; whole-table digest, stats and histo"""
    from oxli_b200.sharded import owner_of

    keys = np.array(sorted(d), dtype=np.uint64)
    vals = np.array([d[int(h)] for h in keys], dtype=np.uint64)
    own = owner_of(keys, world)
    for r, s in enumerate(shards):
        lk, lv = s.local_items_sorted()
        assert np.array_equal(lk, keys[own == r]) and np.array_equal(lv, vals[own == r]), f"rank {r}"
    with np.errstate(over="ignore"):
        want = {"n": len(keys), "sum": int(vals.sum(dtype=np.uint64)), "xor": int(np.bitwise_xor.reduce(keys)) if len(keys) else 0,
                "sum_hc": int((keys * vals).sum(dtype=np.uint64)), "foreign": 0}
    live = [int(v) for v in vals]
    stats = {"len": len(keys), "sum": sum(live) % M64, "min": min(live) if live else 0, "max": max(live) if live else 0}
    hist = {}
    for v in live:
        hist[v] = hist.get(v, 0) + 1
    for got in each_rank(shards, lambda r: (shards[r].digest(), shards[r].stats(), shards[r].engine.histo())):
        assert got[0] == want and got[1] == stats and got[2] == sorted(hist.items())


def consumed_shards(capi, world, k, bases, offs, round_windows=1 << 16):
    from oxli_b200.sharded import ShardedTable, split_reads

    shards = ShardedTable.local(k, world, devices_for(capi, world), round_windows=round_windows)
    n = len(offs) - 1

    def consume(r):
        lo, hi = split_reads(n, r, world)
        shards[r].consume_batch(bases, offs[lo:hi + 1])

    run_ranks([lambda r=r: consume(r) for r in range(world)])
    return shards


@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_add_plain_tables_in_one_process_vs_model(capi, world):
    k = 21 if world % 4 else 31
    bases, offs = reads(71, 16_000)
    d = oracle_dict(k, bases, offs)
    dst_keys = np.array(sorted(d), dtype=np.uint64)
    shards = consumed_shards(capi, world, k, bases, offs)
    Q = shards[0].engine.info()["round_windows"]  # slots of a source per round
    devs = devices_for(capi, world)
    none_rank = 1 if world > 1 else None  # passes None: adds nothing
    rng = np.random.default_rng(world)
    big = [int(h) for h in dst_keys if d[int(h)] >= 3][:2]  # wrap targets: c + 2^64 - 2 and c + 2^64 - 1 stay > 0
    srcs, before = [], []
    for r in range(world):
        if r == none_rank:
            srcs.append(None)
            before.append(None)
            continue
        t = capi.Table(k, devs[r])
        t.reserve(2 * Q)  # >= 4 Q slots: four rounds, most of them empty slots
        assert t.capacity > 2 * Q
        b, o = reads(71, 3000, first_read=100_000 + 3000 * r)  # the same genome: keys shared with dst and the other ranks
        t.consume_batch(b, o)
        special_k = [0, int(rng.integers(1, TOP, dtype=np.uint64)), int(dst_keys[100 + r]), big[0], big[1]]
        special_v = [3 + r, 0, 0, (1 << 64) - 2, (1 << 64) - 1]
        if r in (0, world - 1):
            special_k.append(TOP)
            special_v.append(5 + r)
        if r == 0:  # the wrap targets come from one rank only
            t.add_pairs(special_k, special_v)
        else:
            t.add_pairs(special_k[:3] + special_k[5:], special_v[:3] + special_v[5:])
        srcs.append(t)
        before.append(t.export(1))
    # the model, rank by rank (each zero-valued contribution is the only one to its key, and no sum
    # passes through 0: any order of the additions gives these totals)
    want_added = want_fresh = 0
    for r, e in enumerate(before):
        if e is not None:
            a, f = model_add(d, *e)
            want_added, want_fresh = (want_added + a) % M64, want_fresh + f

    got = each_rank(shards, lambda r: shards[r].add(srcs[r]))
    assert all(g == (want_added, want_fresh) for g in got), (got, want_added, want_fresh)
    check_against(shards, d, world)
    for t, e in zip(srcs, before):
        if t is not None:
            after = t.export(1)
            assert np.array_equal(after[0], e[0]) and np.array_equal(after[1], e[1])
            t.close()
    for s in shards:
        s.close()


@pytest.mark.parametrize("world", [2, 4])
def test_add_sharded_tables(capi, world):
    from oxli_b200.sharded import ShardedTable

    k = 21
    ba, oa = reads(3, 12_000)
    bb, ob = reads(3, 12_000, first_read=50_000)
    A = consumed_shards(capi, world, k, ba, oa)
    B = consumed_shards(capi, world, k, bb, ob)
    da, db = oracle_dict(k, ba, oa), oracle_dict(k, bb, ob)
    b_before = [s.local_items_sorted() for s in B]
    keys = np.array(sorted(db), dtype=np.uint64)
    want = model_add(da, keys, np.array([db[int(h)] for h in keys], dtype=np.uint64))
    got = each_rank(A, lambda r: A[r].add(B[r]))
    assert all(g == want for g in got)
    check_against(A, da, world)
    for s, e in zip(B, b_before):
        after = s.local_items_sorted()
        assert np.array_equal(after[0], e[0]) and np.array_equal(after[1], e[1])
    # another geometry, another k: refused on every rank at once, nothing exchanged
    other = ShardedTable.local(k, world * 2, devices_for(capi, world * 2), round_windows=1 << 16)
    k2 = ShardedTable.local(31, world, devices_for(capi, world), round_windows=1 << 16)
    t0 = time.monotonic()
    for r in range(world):
        assert capi.lib.oxg_shard_merge(A[r].engine._h, other[r].engine._h, None, None) == capi.ERR_INVALID
        assert capi.lib.oxg_shard_merge(A[r].engine._h, k2[r].engine._h, None, None) == capi.ERR_WRONG_KSIZE
        assert capi.lib.oxg_shard_merge(A[r].engine._h, A[r].engine._h, None, None) == capi.ERR_INVALID
        with pytest.raises(ValueError, match="KmerCountTables must have the same ksize"):
            A[r].add(k2[r])
        with pytest.raises(ValueError):
            A[r].add(A[r])
    assert time.monotonic() - t0 < 5
    check_against(A, da, world)
    for s in A + B + other + k2:
        s.close()


def test_consume_add_and_lookup_rounds_interleave(capi):
    from oxli_b200.sharded import split_reads

    world, k = 2, 31
    bases, offs = reads(5, 12_000)
    truth = oracle_dict(k, bases, offs)
    shards = consumed_shards(capi, world, k, bases, offs)
    Q = shards[0].engine.info()["round_windows"]
    devs = devices_for(capi, world)
    d = dict(truth)
    rng = np.random.default_rng(11)
    keys = np.array(sorted(truth), dtype=np.uint64)
    # queries: every key of the reads and of the sources, and random absent ones; more than a round
    srcs = []
    for r in range(world):
        t = capi.Table(k, devs[r])
        b, o = reads(5, 2000, first_read=40_000 + 2000 * r)
        t.consume_batch(b, o)
        t.reserve(Q)
        srcs.append(t)
    src_keys = np.concatenate([t.export(1)[0] for t in srcs])
    q = np.concatenate([keys, src_keys, rng.integers(0, TOP, Q, dtype=np.uint64)])
    rng.shuffle(q)
    queries = [q, q[: len(q) // 3]]

    def expect():
        return [np.array([d.get(int(h), 0) for h in qq], dtype=np.uint64) for qq in queries]

    def again(r):
        lo, hi = split_reads(len(offs) - 1, r, world)
        shards[r].consume_batch(bases, offs[lo:hi + 1])

    for step in range(2):
        if step:  # consume the same reads again
            each_rank(shards, again)
            for h, v in truth.items():
                d[h] = d[h] + v
        for t in srcs:
            model_add(d, *t.export(1))
        each_rank(shards, lambda r: shards[r].add(srcs[r]))
        got = each_rank(shards, lambda r: shards[r].get_hash_array(queries[r]))
        for a, b in zip(got, expect()):
            assert np.array_equal(a, b)
    check_against(shards, d, world)
    for s in shards + srcs:
        s.close()


def test_one_growth_to_what_the_routed_pairs_need(capi):
    from oxli_b200.sharded import ShardedTable, owner_of

    world, k = 2, 21
    devs = devices_for(capi, world)
    shards = ShardedTable.local(k, world, devs, round_windows=1 << 16)
    assert all(s.engine.table.capacity == 1024 for s in shards)
    rng = np.random.default_rng(5)
    # a few keys of its own on every rank
    own = [rng.integers(0, 1 << 63, 100, dtype=np.uint64) | np.uint64(r << 63) for r in range(world)]
    for s, o in zip(shards, own):
        s.engine.table.count_hashes(o)
    n_src = 2_000_000
    srcs, pairs = [], []
    for r in range(world):
        kk = np.unique(rng.integers(0, TOP, n_src + 1000, dtype=np.uint64))[:n_src]
        kk = kk[kk != np.uint64(TOP)]
        vv = rng.integers(1, 1000, len(kk), dtype=np.uint64)
        t = capi.Table(k, devs[r])
        t.add_pairs(kk, vv)
        srcs.append(t)
        pairs.append((kk, vv))
    allk = np.concatenate([p[0] for p in pairs] + own)
    routed = [int(np.count_nonzero(owner_of(np.concatenate([p[0] for p in pairs]), world) == r)) for r in range(world)]
    each_rank(shards, lambda r: shards[r].add(srcs[r]))
    for r, s in enumerate(shards):
        scratch = capi.Table(k, devs[r])
        scratch.reserve(len(own[r]) + routed[r])
        assert s.engine.table.capacity == scratch.capacity
        scratch.close()
    # exact: the model by sorting (keys of different ranks may coincide: their counts add)
    vals = np.concatenate([p[1] for p in pairs] + [np.ones(len(o), dtype=np.uint64) for o in own])
    uk, inv = np.unique(allk, return_inverse=True)
    uv = np.zeros(len(uk), dtype=np.uint64)
    np.add.at(uv, inv, vals)
    o = owner_of(uk, world)
    for r, s in enumerate(shards):
        lk, lv = s.local_items_sorted()
        assert np.array_equal(lk, uk[o == r]) and np.array_equal(lv, uv[o == r])
    for s in shards + srcs:
        s.close()


def test_skewed_source_all_to_owner_zero(capi):
    world, k = 4, 21
    bases, offs = reads(9, 8000)
    d = oracle_dict(k, bases, offs)
    shards = consumed_shards(capi, world, k, bases, offs)
    devs = devices_for(capi, world)
    rng = np.random.default_rng(9)
    srcs = []
    for r in range(world):
        kk = rng.integers(0, 1 << 62, 300_000, dtype=np.uint64)  # owner 0 of 4: the top two bits are 0
        kk[:1000] = np.array(sorted(d), dtype=np.uint64)[:1000]  # (the smallest keys of dst: owner 0 as well)
        t = capi.Table(k, devs[r])
        t.count_hashes(kk)
        srcs.append(t)
    for t in srcs:
        model_add(d, *t.export(1))
    each_rank(shards, lambda r: shards[r].add(srcs[r]))
    check_against(shards, d, world)
    for s in shards + srcs:
        s.close()


def _merge_worker(rank, world, k, conns, out_dir):
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
    n = 16_000
    bases = synth_reads(n, L, G, seed=13, n_ppm=500)
    offs = uniform_offsets(n, L)
    t = ShardedTable(k, rank, world, device=dev, exchange=exchange, round_windows=1 << 16)
    lo, hi = split_reads(n, rank, world)
    t.consume_batch(bases, offs[lo:hi + 1])
    src = capi.Table(k, dev)
    src.consume_batch(synth_reads(3000, L, G, seed=13, first_read=30_000 + 3000 * rank, n_ppm=500), uniform_offsets(3000, L))
    src.add_pairs([TOP, 0], [2 + rank, 1])
    src.reserve(2 * t.engine.info()["round_windows"])
    sk, sv = src.export(1)
    totals = t.add(src)
    lk, lv = t.local_items_sorted()
    np.savez(os.path.join(out_dir, f"merge{rank}.npz"), sk=sk, sv=sv, lk=lk, lv=lv, totals=np.array(totals, dtype=np.uint64))
    exchange(b"done")  # nobody unmaps an exchange area a peer may still be reading
    src.close()
    t.close()


def test_add_in_separate_processes_over_cuda_ipc(capi, tmp_path):
    import multiprocessing as mp

    from oxli_b200.sharded import owner_of

    world, k = 2, 31
    ctx = mp.get_context("spawn")
    a, b = ctx.Pipe()
    procs = [ctx.Process(target=_merge_worker, args=(0, world, k, [a], str(tmp_path))),
             ctx.Process(target=_merge_worker, args=(1, world, k, b, str(tmp_path)))]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    d = oracle_dict(k, synth_reads(16_000, L, G, seed=13, n_ppm=500), uniform_offsets(16_000, L))
    parts = [np.load(tmp_path / f"merge{r}.npz") for r in range(world)]
    added = fresh = 0
    for p in parts:
        a_, f_ = model_add(d, p["sk"], p["sv"])
        added, fresh = (added + a_) % M64, fresh + f_
    keys = np.array(sorted(d), dtype=np.uint64)
    vals = np.array([d[int(h)] for h in keys], dtype=np.uint64)
    own = owner_of(keys, world)
    for r, p in enumerate(parts):
        assert np.array_equal(p["lk"], keys[own == r]) and np.array_equal(p["lv"], vals[own == r])
        assert p["totals"].tolist() == [added, fresh]


def test_refused_calls_start_no_exchange(capi):
    from oxli_b200.sharded import ShardedTable

    lib = capi.lib
    s = capi.Shard(21, 0, 1)
    s.table.count_hashes([5, 5, 9])
    d0 = s.digest()
    t31 = capi.Table(31)
    t31.count_hashes([1, 2])
    assert lib.oxg_shard_merge_table(s._h, t31._h, None, None) == capi.ERR_WRONG_KSIZE
    assert b"KmerCountTables must have the same ksize" in lib.oxg_last_error()
    assert lib.oxg_shard_merge_table(s._h, s.table._h, None, None) == capi.ERR_INVALID
    assert s.digest() == d0
    assert s.merge_table(None) == (0, 0) and s.digest() == d0
    t21 = capi.Table(21)
    t21.count_hashes([5, 7])
    assert s.merge_table(t21) == (2, 1) and s.get_hashes([5, 7, 9]).tolist() == [3, 1, 1]
    s.close()
    lone = capi.Shard(21, 0, 2)  # peers not connected: refused at once
    assert lib.oxg_shard_merge_table(lone._h, t21._h, None, None) == capi.ERR_INVALID
    assert b"not connected" in lib.oxg_last_error()
    lone.close()
    # a refused call on one rank of a connected pair returns at once: had it started an exchange,
    # it would have waited for the other rank; both ranks then add together as usual
    pair = ShardedTable.local(21, 2, devices_for(capi, 2))
    d1 = each_rank(pair, lambda r: pair[r].digest())[0]
    t0 = time.monotonic()
    assert lib.oxg_shard_merge_table(pair[0].engine._h, t31._h, None, None) == capi.ERR_WRONG_KSIZE
    assert lib.oxg_shard_merge_table(pair[0].engine._h, pair[0].engine.table._h, None, None) == capi.ERR_INVALID
    with pytest.raises(ValueError, match="KmerCountTables must have the same ksize"):
        pair[0].add(t31)
    with pytest.raises(ValueError):
        pair[0].add(pair[0].engine.table)
    assert time.monotonic() - t0 < 5
    assert each_rank(pair, lambda r: pair[r].digest())[0] == d1
    got = each_rank(pair, lambda r: pair[r].add(t21 if r == 0 else None))
    assert got == [(2, 2), (2, 2)]
    assert each_rank(pair, lambda r: pair[r].get_hash_array([5, 7]).tolist()) == [[1, 1], [1, 1]]
    for p in pair:
        p.close()
    t21.close()
    t31.close()


def test_source_on_another_device_is_refused(capi):
    if capi.lib.oxg_device_count() < 2:
        pytest.skip("needs a second GPU")
    s = capi.Shard(21, 0, 1, device=0)
    s.table.count_hashes([5])
    d0 = s.digest()
    t = capi.Table(21, device=1)
    t.count_hashes([5])
    assert capi.lib.oxg_shard_merge_table(s._h, t._h, None, None) == capi.ERR_INVALID
    assert s.digest() == d0
    t.close()
    s.close()
