"""Export and dump of the hash-sharded table (oxg_shard_export_pairs, oxg_shard_dump;
ShardedTable.export / dump, src/lib.rs:330-381) against a plain table holding the same pairs.

Every key of rank r is below every key of rank r + 1, so each rank sorts and formats its own shard
and writes its part of one file.  The model of each result is a plain `_capi.Table` built from the
same pairs, its export(mode) formatted as the reference's dump lines; one case compares with the
drop-in KmerCountTable.dump file itself.  As in test_gpu_shard_lookup.py, several shards on one GPU
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
FLAGS = {0: {}, 1: {"sortkeys": True}, 2: {"sortcounts": True}}


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


def each_rank(shards, fn):
    """fn(r) on every rank at once (collective calls); returns the results in rank order"""
    out = [None] * len(shards)

    def go(r):
        out[r] = fn(r)

    run_ranks([lambda r=r: go(r) for r in range(len(shards))])
    return out


def devices_for(capi, world):
    n = capi.lib.oxg_device_count()
    return [r % n for r in range(world)]


def reads(seed, n):
    return synth_reads(n, L, G, seed=seed, sub_ppm=5000, n_ppm=800), uniform_offsets(n, L)


def consumed_shards(capi, world, k, bases, offs):
    from oxli_b200.sharded import ShardedTable

    shards = ShardedTable.local(k, world, devices_for(capi, world), round_windows=1 << 16)
    consume_again(shards, bases, offs)
    return shards


def consume_again(shards, bases, offs):
    from oxli_b200.sharded import split_reads

    n, world = len(offs) - 1, len(shards)

    def consume(r):
        lo, hi = split_reads(n, r, world)
        shards[r].consume_batch(bases, offs[lo:hi + 1])

    run_ranks([lambda r=r: consume(r) for r in range(world)])


def text(keys, vals) -> bytes:
    return "".join(f"{k}\t{v}\n" for k, v in zip(np.asarray(keys).tolist(), np.asarray(vals).tolist())).encode()


def all_pairs(shards):
    """every rank's pairs (plain-table export of its shard, not the code under test)"""
    parts = [s.engine.table.export(0) for s in shards]
    return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])


def plain_model(capi, k, keys, vals, device=0):
    """a plain table holding the same pairs: its export in each sort mode"""
    t = capi.Table(k, device)
    t.add_pairs(keys, vals)
    assert len(t) == len(keys)
    out = {m: t.export(m) for m in (0, 1, 2)}
    t.close()
    return out


def assemble(parts):
    """the whole table from every rank's (keys, vals, runs, total): runs applied in order"""
    total = parts[0][3]
    assert all(p[3] == total for p in parts)
    K = np.zeros(total, dtype=np.uint64)
    V = np.zeros(total, dtype=np.uint64)
    seen = np.zeros(total, dtype=np.int64)
    for k, v, runs, _ in parts:
        pos = 0
        for start, length in runs.tolist():
            K[start:start + length] = k[pos:pos + length]
            V[start:start + length] = v[pos:pos + length]
            seen[start:start + length] += 1
            pos += length
        assert pos == len(k)
    assert (seen == 1).all()
    return K, V


def check_mode0(shards, parts, K, V, mk, mv):
    """slot order: the same multiset, each rank's shard in one block, the blocks in rank order"""
    from oxli_b200.sharded import owner_of

    before = 0
    for r, (k, _, runs, _) in enumerate(parts):
        assert runs.tolist() == [[before, len(k)]]
        before += len(k)
        assert (owner_of(k, len(shards)) == r).all()
    a, b = np.lexsort((V, K)), np.lexsort((mv, mk))
    assert np.array_equal(K[a], mk[b]) and np.array_equal(V[a], mv[b])


def check_export_and_dump(capi, shards, tmp_path, k, model=None, tag=""):
    """export and dump in every mode against the plain-table model of the same pairs"""
    if model is None:
        model = plain_model(capi, k, *all_pairs(shards))
    for mode, flags in FLAGS.items():
        parts = each_rank(shards, lambda r: shards[r].export(**flags))
        K, V = assemble(parts)
        mk, mv = model[mode]
        path = str(tmp_path / f"dump{tag}_{mode}.tsv")
        each_rank(shards, lambda r: shards[r].dump(path, **flags))
        got = open(path, "rb").read()
        if mode == 0:
            check_mode0(shards, parts, K, V, mk, mv)
            assert got == text(K, V)  # the file holds the lines of the assembled slot-order export
            assert sorted(got.splitlines()) == sorted(text(mk, mv).splitlines())
        else:
            assert np.array_equal(K, mk) and np.array_equal(V, mv), mode
            assert got == text(mk, mv), mode
        assert os.path.getsize(path) == len(text(mk, mv))
        os.remove(path)
    return model


# ---- 1. consumed tables, N = 1, 2, 4, 8 ---------------------------------------------------------

@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_export_and_dump_vs_plain_table(capi, world, tmp_path):
    k = 21 if world % 4 else 31
    bases, offs = reads(90 + world, 16_000)
    shards = consumed_shards(capi, world, k, bases, offs)
    shards[world - 1].engine.table.set_hash(TOP, 7)  # 2^64-1 lives in its owner's side entry
    shards[0].engine.table.set_hash(5, 0)            # a key held with count 0
    check_export_and_dump(capi, shards, tmp_path, k)
    for s in shards:
        s.close()


def test_dump_matches_the_dropin_dump_file(capi, tmp_path):
    """the bytes of the drop-in KmerCountTable.dump of the same reads (modes 1 and 2), its lines (mode 0)"""
    from oxli_b200 import KmerCountTable

    world, k = 2, 21
    bases, offs = reads(7, 12_000)
    shards = consumed_shards(capi, world, k, bases, offs)
    ref = KmerCountTable(k)
    ref.consume_buffer(bases, offs, True)
    assert len(ref) == each_rank(shards, lambda r: len(shards[r]))[0]
    for mode, flags in FLAGS.items():
        mine, theirs = str(tmp_path / f"sharded{mode}.tsv"), str(tmp_path / f"dropin{mode}.tsv")
        each_rank(shards, lambda r: shards[r].dump(mine, **flags))
        ref.dump(theirs, **flags)
        a, b = open(mine, "rb").read(), open(theirs, "rb").read()
        assert (a == b) if mode else (sorted(a.splitlines()) == sorted(b.splitlines()))
    for s in shards:
        s.close()


# ---- 2. crafted tables ----------------------------------------------------------------------------

def digit_edges():
    """0, 1, 9, 10, 99, 100, ..., 10^19, 2^64-2, 2^64-1: every decimal length on both sides"""
    out = {0, TOP, TOP - 1}
    for d in range(1, 21):
        out.add(10 ** (d - 1))
        out.add(min(10 ** d - 1, TOP))
    return sorted(out)


def crafted_shards(capi, world, pairs_of_rank, k=21):
    """fresh shards; rank r adds its plain table of pairs_of_rank[r] (keys of any owner)"""
    from oxli_b200.sharded import ShardedTable

    devs = devices_for(capi, world)
    shards = ShardedTable.local(k, world, devs, round_windows=1 << 16)
    srcs = []
    for r in range(world):
        t = capi.Table(k, devs[r])
        kk, vv = pairs_of_rank[r]
        if len(kk):
            t.add_pairs(kk, vv)
        srcs.append(t)
    each_rank(shards, lambda r: shards[r].add(srcs[r]))
    for t in srcs:
        t.close()
    return shards


def test_crafted_digits_zero_counts_an_empty_rank_and_many_counts(capi, tmp_path):
    """keys and counts of every decimal length (0 and 2^64-1 included), rank 1 owning nothing, more
    than 65 536 distinct counts on rank 0 (its per-count blocks and its histogram cross several
    all-gather pieces) and 4 M keys on rank 3 (its text crosses several chunk boundaries)"""
    from oxli_b200.sharded import owner_of

    world = 4
    rng = np.random.default_rng(12)
    edges = np.array(digit_edges(), dtype=np.uint64)
    edge_counts = edges[::-1].copy()  # 0 and 2^64-1 among them (2^64-1 held with count 0)
    many = np.unique(rng.integers(1, 1 << 62, 90_000, dtype=np.uint64))[:80_000]     # rank 0
    many_counts = rng.permutation(np.arange(80_000, dtype=np.uint64) * np.uint64(104_729) + np.uint64(3))
    bulk = np.unique(rng.integers(3 << 62, TOP - 1, 4_100_000, dtype=np.uint64))[:4_000_000]  # rank 3
    bulk_counts = rng.integers(0, 6, len(bulk), dtype=np.uint64)
    keys = np.concatenate([edges, many, bulk])
    vals = np.concatenate([edge_counts, many_counts, bulk_counts])
    keys, first = np.unique(keys, return_index=True)
    vals = vals[first]
    keep = owner_of(keys, world) != 1
    keys, vals = keys[keep], vals[keep]
    assert len(np.unique(vals[owner_of(keys, world) == 0])) > 65_536
    order = rng.permutation(len(keys))  # every rank adds a slice of keys of every owner
    pairs = [(keys[order[r::world]], vals[order[r::world]]) for r in range(world)]
    shards = crafted_shards(capi, world, pairs)
    assert len(shards[1].engine.table) == 0
    n3 = len(shards[3].engine.table)
    rw = shards[3].engine.info()["round_windows"]
    assert n3 > 4 * (min(rw, 4 << 20) // 1024 * 1024)  # five chunks of text on rank 3 (the fewest pairs a round holds: 0.9 Mi on a B200)
    model = check_export_and_dump(capi, shards, tmp_path, 21)
    assert model[2][1][0] == 0 and model[2][1][-1] == TOP and model[1][0][-1] == TOP
    freq, n = np.unique(model[2][1], return_counts=True)  # the sparse histogram of every count
    assert each_rank(shards, lambda r: shards[r].engine.histo()) == [list(zip(freq.tolist(), n.tolist()))] * world
    for s in shards:
        s.close()


@pytest.mark.parametrize("world", [1, 2])
def test_empty_table_dumps_an_empty_file(capi, world, tmp_path):
    from oxli_b200.sharded import ShardedTable

    shards = ShardedTable.local(21, world, devices_for(capi, world), round_windows=1 << 16)
    for mode, flags in FLAGS.items():
        parts = each_rank(shards, lambda r: shards[r].export(**flags))
        for k, v, runs, total in parts:
            assert total == 0 and len(k) == 0 and runs.tolist() == ([] if mode == 2 else [[0, 0]])
        path = tmp_path / f"empty{mode}.tsv"
        path.write_bytes(b"left over")  # truncated
        each_rank(shards, lambda r: shards[r].dump(str(path), **flags))
        assert path.read_bytes() == b""
    for s in shards:
        s.close()


# ---- 3. two processes -------------------------------------------------------------------------------

def _dump_worker(rank, world, k, conns, out_dir):
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
    n = 20_000
    bases = synth_reads(n, L, 120_000, seed=17, n_ppm=500)
    offs = uniform_offsets(n, L)
    t = ShardedTable(k, rank, world, device=dev, exchange=exchange, round_windows=1 << 16)
    lo, hi = split_reads(n, rank, world)
    t.consume_batch(bases, offs[lo:hi + 1])
    if rank == world - 1:
        t.engine.table.set_hash(TOP, 4)
    for mode, flags in FLAGS.items():
        t.dump(os.path.join(out_dir, f"ipc{mode}.tsv"), **flags)
    k_, v_ = t.engine.table.export(0)
    np.savez(os.path.join(out_dir, f"ipc{rank}.npz"), keys=k_, vals=v_)
    exchange(b"done")  # nobody unmaps an exchange area a peer may still be reading
    t.close()


def test_dump_from_separate_processes_over_cuda_ipc(capi, tmp_path):
    import multiprocessing as mp

    world, k = 2, 31
    ctx = mp.get_context("spawn")
    a, b = ctx.Pipe()
    procs = [ctx.Process(target=_dump_worker, args=(0, world, k, [a], str(tmp_path))),
             ctx.Process(target=_dump_worker, args=(1, world, k, b, str(tmp_path)))]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    parts = [np.load(tmp_path / f"ipc{r}.npz") for r in range(world)]
    keys = np.concatenate([p["keys"] for p in parts])
    vals = np.concatenate([p["vals"] for p in parts])
    truth = OracleTable(k)  # the pairs themselves against the oracle
    truth.consume_batch(synth_reads(20_000, L, 120_000, seed=17, n_ppm=500), uniform_offsets(20_000, L), True, nthreads=4)
    tk, tv = truth.items_sorted()
    d = dict(zip(tk.tolist(), tv.tolist()))
    d[TOP] = 4
    assert dict(zip(keys.tolist(), vals.tolist())) == d
    model = plain_model(capi, k, keys, vals)
    assert (tmp_path / "ipc1.tsv").read_bytes() == text(*model[1])
    assert (tmp_path / "ipc2.tsv").read_bytes() == text(*model[2])
    got0 = (tmp_path / "ipc0.tsv").read_bytes()
    assert got0 == text(parts[0]["keys"], parts[0]["vals"]) + text(parts[1]["keys"], parts[1]["vals"])


# ---- 4. among the other collective calls --------------------------------------------------------------

def oracle_dict(k, bases, offs):
    t = OracleTable(k)
    t.consume_batch(bases, offs, True, nthreads=4)
    tk, tv = t.items_sorted()
    return dict(zip(tk.tolist(), tv.tolist()))


def dict_model(d):
    keys = np.array(sorted(d), dtype=np.uint64)
    vals = np.array([d[int(h)] for h in keys.tolist()], dtype=np.uint64)
    order = np.lexsort((keys, vals))
    return {1: (keys, vals), 2: (keys[order], vals[order])}


def dump_matches(shards, d, path, mode):
    each_rank(shards, lambda r: shards[r].dump(path, **FLAGS[mode]))
    return open(path, "rb").read() == text(*dict_model(d)[mode])


def test_dump_and_export_between_consume_lookup_merge_and_erase(capi, tmp_path):
    """consume -> dump -> lookup -> export -> merge -> dump -> erase -> export -> consume, against a
    dict model: a dump or an export changes nothing the other calls see"""
    world, k = 2, 21
    bases, offs = reads(5, 12_000)
    counts = oracle_dict(k, bases, offs)
    d = dict(counts)
    shards = consumed_shards(capi, world, k, bases, offs)
    devs = devices_for(capi, world)
    path = str(tmp_path / "between.tsv")
    assert dump_matches(shards, d, path, 2)
    keys = np.array(sorted(d), dtype=np.uint64)
    q = [keys[r::5] for r in range(world)]
    got = each_rank(shards, lambda r: shards[r].get_hash_array(q[r]))
    for a, b in zip(q, got):
        assert b.tolist() == [d.get(int(h), 0) for h in a.tolist()]
    K, V = assemble(each_rank(shards, lambda r: shards[r].export(sortkeys=True)))
    assert np.array_equal(K, dict_model(d)[1][0]) and np.array_equal(V, dict_model(d)[1][1])
    rng = np.random.default_rng(4)
    srcs = []
    for r in range(world):  # (made before the ranks start: allocations synchronise the device)
        t = capi.Table(k, devs[r])
        sk = np.unique(np.concatenate([keys[r::7], rng.integers(0, TOP, 1000, dtype=np.uint64)]))
        t.add_pairs(sk, np.full(len(sk), 2 + r, dtype=np.uint64))
        srcs.append(t)
        for h in sk.tolist():
            d[h] = d.get(h, 0) + 2 + r
    each_rank(shards, lambda r: shards[r].add(srcs[r]))
    assert dump_matches(shards, d, path, 1)
    gone = [keys[:300], keys[-300:]]
    each_rank(shards, lambda r: shards[r].drop_hash_array(gone[r]))
    for lst in gone:
        for h in lst.tolist():
            d.pop(h, None)
    K, V = assemble(each_rank(shards, lambda r: shards[r].export(sortcounts=True)))
    assert np.array_equal(K, dict_model(d)[2][0]) and np.array_equal(V, dict_model(d)[2][1])
    consume_again(shards, bases, offs)
    for h, c in counts.items():
        d[h] = d.get(h, 0) + c
    keys = np.array(sorted(d), dtype=np.uint64)
    vals = np.array([d[int(h)] for h in keys.tolist()], dtype=np.uint64)
    with np.errstate(over="ignore"):
        want = {"n": len(keys), "sum": int(vals.sum(dtype=np.uint64)), "xor": int(np.bitwise_xor.reduce(keys)),
                "sum_hc": int((keys * vals).sum(dtype=np.uint64)), "foreign": 0}
    assert each_rank(shards, lambda r: shards[r].digest()) == [want, want]
    assert dump_matches(shards, d, path, 2)
    for t in srcs:
        t.close()
    for s in shards:
        s.close()


# ---- 5. refusals and file errors ------------------------------------------------------------------------

def test_refused_calls_start_no_exchange(capi, tmp_path):
    from oxli_b200.sharded import ShardedTable

    lib, err_invalid = capi.lib, capi.ERR_INVALID
    n = capi.u64()
    path = str(tmp_path / "refused.tsv").encode()
    lone = capi.Shard(21, 0, 2)  # a shard whose peers are not connected: refused at once
    assert lib.oxg_shard_dump(lone._h, path, 1) == err_invalid
    assert b"not connected" in lib.oxg_last_error()
    assert lib.oxg_shard_export_pairs(lone._h, 1, None, None, 0, n, None, 0, n, n) == err_invalid
    lone.close()
    pair = ShardedTable.local(21, 2, devices_for(capi, 2))
    pair[0].engine.table.count_hashes([5, 5, 9])
    pair[1].engine.table.set_hash(TOP, 3)
    buf = np.zeros(4, dtype=np.uint64)
    h = pair[0].engine._h
    # refused on rank 0 alone: had it started an exchange, it would have waited for rank 1
    for call in (lambda: lib.oxg_shard_dump(h, None, 1),
                 lambda: lib.oxg_shard_dump(h, path, 3),
                 lambda: lib.oxg_shard_dump(h, path, -1),
                 lambda: lib.oxg_shard_export_pairs(h, 3, None, None, 0, n, None, 0, n, n),
                 lambda: lib.oxg_shard_export_pairs(h, 1, None, None, 4, n, None, 0, n, n),
                 lambda: lib.oxg_shard_export_pairs(h, 1, buf.ctypes.data, buf.ctypes.data, 4, n, None, 2, n, n)):
        t0 = time.monotonic()
        assert call() == err_invalid
        assert time.monotonic() - t0 < 5
    assert not os.path.exists(path)
    # ranks that pass different paths: a collective failure, the same on both ranks, no file
    paths = [str(tmp_path / "a.tsv"), str(tmp_path / "b.tsv")]
    for r, e in enumerate(each_rank(pair, lambda r: _raised(lambda: pair[r].dump(paths[r], sortkeys=True)))):
        assert isinstance(e, capi.OxliError) and e.status == err_invalid and "different paths" in str(e), (r, e)
    assert not any(os.path.exists(p) for p in paths)
    # both ranks then dump together as usual
    each_rank(pair, lambda r: pair[r].dump(path.decode(), sortcounts=True))
    assert open(path, "rb").read() == b"9\t1\n5\t2\n" + f"{TOP}\t3\n".encode()
    for p in pair:
        p.close()


def _raised(fn):
    try:
        fn()
    except Exception as e:  # noqa: BLE001
        return e
    return None


def test_a_missing_directory_raises_oserror_on_every_rank_promptly(capi, tmp_path):
    world, k = 2, 21
    bases, offs = reads(3, 4_000)
    shards = consumed_shards(capi, world, k, bases, offs)
    bad = str(tmp_path / "no_such_dir" / "counts.tsv")
    t0 = time.monotonic()
    errs = each_rank(shards, lambda r: _raised(lambda: shards[r].dump(bad, sortkeys=True)))
    assert time.monotonic() - t0 < 10  # far inside the 30 s a peer waits before it gives up
    for r, e in enumerate(errs):
        assert isinstance(e, OSError), (r, e)
    assert "no_such_dir" in str(errs[0]) and "rank 0" in str(errs[1])
    check_export_and_dump(capi, shards, tmp_path, k)  # the table is as usable as before
    for s in shards:
        s.close()
