"""Removing keys from the hash-sharded table (oxg_shard_erase_hashes*, oxg_shard_cut;
ShardedTable.drop / drop_hash / drop_hash_array / mincut / maxcut) against a host model built with
the oracle (src/lib.rs:197-267).

Every rank passes its own list; each key goes to the rank that owns it, in exchange rounds of the
same kind as consume, lookup and merge rounds, and is erased there: in place for fewer than 256 keys
over all ranks, else by marking slots and one rebuild per owner.  After every call each rank's
contents, the whole-table digest, stats and histogram, the removed count (the same on every rank)
and lookups of the dropped keys are checked.  As in test_gpu_shard_lookup.py, several shards on one
GPU run the same code as one shard per GPU."""
import os
import random
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
PHI = 0x9E3779B97F4A7C15
PHI_INV = pow(PHI, -1, M64)
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


def reads(seed, n):
    return synth_reads(n, L, G, seed=seed, sub_ppm=5000, n_ppm=800), uniform_offsets(n, L)


def oracle_dict(k, bases, offs):
    t = OracleTable(k)
    t.consume_batch(bases, offs, True, nthreads=4)
    tk, tv = t.items_sorted()
    return dict(zip(tk.tolist(), tv.tolist()))


def consumed_shards(capi, world, k, bases, offs, round_windows=1 << 16):
    from oxli_b200.sharded import ShardedTable

    shards = ShardedTable.local(k, world, devices_for(capi, world), round_windows=round_windows)
    consume_again(shards, bases, offs)
    return shards


def consume_again(shards, bases, offs):
    from oxli_b200.sharded import split_reads

    n, world = len(offs) - 1, len(shards)

    def consume(r):
        lo, hi = split_reads(n, r, world)
        shards[r].consume_batch(bases, offs[lo:hi + 1])

    run_ranks([lambda r=r: consume(r) for r in range(world)])


def model_drop(d, lists):
    """drop_hash of every listed key from dict d: the distinct keys removed"""
    gone = {int(h) for lst in lists for h in np.asarray(lst, dtype=np.uint64).tolist()} & set(d)
    for h in gone:
        del d[h]
    return len(gone)


def check_against(shards, d):
    """every rank holds exactly its owner's slice of d; whole-table digest, stats and histo"""
    from oxli_b200.sharded import owner_of

    world = len(shards)
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


def dropped_with_launches(shards, lists):
    """every rank drops its list; returns what each rank was told, and the kernel launches the
    collective call took over all ranks"""
    from oxli_b200 import _capi

    before = _capi.lib.oxg_launch_count()
    got = each_rank(shards, lambda r: shards[r].drop_hash_array(lists[r]))
    return got, _capi.lib.oxg_launch_count() - before


def drop_and_check(shards, lists, d, launches=None):
    """every rank drops its list; the model drops them all; totals, contents and lookups agree.
    launches (if given) receives the kernel launches of the drop."""
    want = model_drop(d, lists)
    got, n_launches = dropped_with_launches(shards, lists)
    if launches is not None:
        launches.append(n_launches)
    assert got == [want] * len(shards), (got, want)
    check_against(shards, d)
    answers = each_rank(shards, lambda r: shards[r].get_hash_array(lists[r]))
    for lst, a in zip(lists, answers):
        assert a.tolist() == [d.get(int(h), 0) for h in np.asarray(lst, dtype=np.uint64).tolist()]
    return want


def make_list(rng, keys, size, extra=()):
    """half present keys (drawn with replacement: duplicates), half random u64 (absent), plus 0,
    the given extras and repeats, shuffled"""
    if size == 0:
        return np.zeros(0, dtype=np.uint64)
    n_present = size // 2
    present = keys[rng.integers(0, len(keys), n_present)]
    absent = rng.integers(0, TOP, size - n_present, dtype=np.uint64, endpoint=True)
    q = np.concatenate([present, absent, np.array([0, *extra], dtype=np.uint64), present[:4]])
    rng.shuffle(q)
    return q


# ---- 1. lists over several rounds (mark and rebuild) --------------------------------------------

# "staged": rounds of 2.5 Mi keys, so that rank 0's host list crosses in several pieces of the
# shard's 1 Mi-entry staging buffer per round, the last of them partly filled
@pytest.mark.parametrize("world,round_windows", [(1, 1 << 16), (2, 1 << 16), (4, 1 << 16), (8, 1 << 16), (4, 5 << 19)],
                         ids=["1", "2", "4", "8", "4-staged"])
def test_drop_lists_in_one_process_vs_model(capi, world, round_windows):
    from oxli_b200.sharded import owner_of

    k = 21 if world % 4 else 31
    bases, offs = reads(71, 16_000)
    d = oracle_dict(k, bases, offs)
    shards = consumed_shards(capi, world, k, bases, offs, round_windows)
    shards[world - 1].engine.table.set_hash(TOP, 7)  # 2^64-1 lives in its owner's side entry
    d[TOP] = 7
    Q = shards[0].engine.info()["round_windows"]  # keys per rank and round
    assert Q >= round_windows
    keys = np.array(sorted(d), dtype=np.uint64)
    rng = np.random.default_rng(world)
    # rank 0 needs three rounds, the others less, rank 1 nothing; 2^64-1 from rank 0 and the last
    # rank at once; keys of rank 0's list repeated by the others
    sizes = [2 * Q + 1] + [0 if r == 1 else Q // (2 * r) + r for r in range(1, world)]
    lists = [make_list(rng, keys, s, extra=(TOP,) if r in (0, world - 1) else ()) for r, s in enumerate(sizes)]
    for r in range(2, world):
        lists[r] = np.concatenate([lists[r], lists[0][:500]])
    assert set(owner_of(lists[0], world).tolist()) == set(range(world))
    assert drop_and_check(shards, lists, d) > len(keys) // 4
    assert TOP not in d
    # again: 2^64-1 and the dropped keys are absent now; some keys still present go
    lists = [np.concatenate([lst[: len(lst) // 2], keys[r::97], np.array([TOP], dtype=np.uint64)]) for r, lst in enumerate(lists)]
    assert drop_and_check(shards, lists, d) > 0
    for s in shards:
        s.close()


# ---- 2 and 3. few keys (in place), runs that wrap and long runs ---------------------------------

def lg_of(cap):
    return cap.bit_length() - 1


def home(key, cap):
    return (((key * PHI) % M64) >> (64 - lg_of(cap))) & ~1


def keys_homed(slot, cap, n, rr, taken, accept):
    """n new keys homed at the even `slot` of a table of `cap` slots, owned as accept() says"""
    out = []
    while len(out) < n:
        key = (((slot << (64 - lg_of(cap))) | rr.getrandbits(64 - lg_of(cap))) * PHI_INV) % M64
        if key != TOP and key not in taken and accept(key):
            taken.add(key)
            out.append(key)
    return out


def cluster(n, top40, accept):
    """n keys whose key * PHI share the top 40 bits: one home at every capacity"""
    out, low = [], 0
    while len(out) < n:
        key = (((top40 << 24) | low) * PHI_INV) % M64
        low += 1
        if key != TOP and accept(key):
            out.append(key)
    return out


class SlotModel:
    """a slot array filled one key at a time (set_hash), emptied one key at a time: linear probing
    from home(key), erase by backward shift"""

    def __init__(self, cap):
        self.cap, self.slots, self.side = cap, {}, None

    def find(self, key):
        i = home(key, self.cap)
        while i in self.slots:
            if self.slots[i][0] == key:
                return i
            i = (i + 1) % self.cap
        return None

    def set(self, key, v):
        if key == TOP:
            self.side = v
            return
        i = self.find(key)
        if i is None:
            i = home(key, self.cap)
            while i in self.slots:
                i = (i + 1) % self.cap
        self.slots[i] = (key, v)

    def erase(self, key):
        if key == TOP:
            had, self.side = self.side is not None, None
            return int(had)
        hole = self.find(key)
        if hole is None:
            return 0
        del self.slots[hole]
        j = hole
        while True:
            j = (j + 1) % self.cap
            if j not in self.slots:
                return 1
            if (j - home(self.slots[j][0], self.cap)) % self.cap >= (j - hole) % self.cap:
                self.slots[hole] = self.slots.pop(j)
                hole = j

    def export(self):
        """what export(0) gives: slot order, then the side entry"""
        out = [self.slots[i] for i in sorted(self.slots)]
        return out + ([(TOP, self.side)] if self.side is not None else [])

    def items(self):
        return dict(self.export())


def crafted_shards(capi, seed, cap=1 << 14):
    """two fresh shards on one GPU, each holding keys it owns (top bit = rank), set one at a time:
    a run across slot cap-1 -> 0, an 800-key run at cap/2, random keys.  Returns the shards, their
    slot models, the runs and absent keys homed in them."""
    from oxli_b200.sharded import ShardedTable

    world = 2
    shards = ShardedTable.local(21, world, devices_for(capi, world), capacity_hint=cap * 3 // 10, round_windows=1 << 16)
    rr = random.Random(seed)
    models, runs, probes, taken = [], [], [], set()
    for r, s in enumerate(shards):
        t = s.engine.table
        assert t.capacity == cap  # the capacity the keys are made for
        own = (lambda r: lambda key: key >> 63 == r)(r)
        wrap = [key for h, n in ((-4, 5), (-2, 6), (0, 4), (2, 3)) for key in keys_homed(h % cap, cap, n, rr, taken, own)]
        run = cluster(900, (cap // 2) << (40 - lg_of(cap)), own)
        taken |= set(run)
        rand = [key for _ in range(100) for key in keys_homed(2 * rr.randrange(cap // 2), cap, 1, rr, taken, own)]
        m = SlotModel(cap)
        for i, key in enumerate(wrap + run[:800] + rand):
            t.set_hash(key, i % 50 + 1)
            m.set(key, i % 50 + 1)
        assert all(sl in m.slots for sl in list(range(cap - 4, cap)) + list(range(0, 8)))  # the run wraps
        assert all(cap // 2 + i in m.slots for i in range(800))
        k, v = t.export(0)
        assert list(zip(k.tolist(), v.tolist())) == m.export()
        models.append(m)
        runs.append((wrap, run[:800]))
        probes += run[800:] + [key for sl in (cap - 4, cap - 2, 0, 2) for key in keys_homed(sl, cap, 2, rr, taken, own)]
    return shards, models, runs, probes


def test_few_keys_are_erased_in_place_across_the_wrap_and_in_long_runs(capi):
    """fewer than 256 keys over all ranks: each owner erases in place by backward shift; its
    slot-order export matches the model slot for slot, so no rebuild ran"""
    shards, models, runs, probes = crafted_shards(capi, 80)
    cap = models[0].cap

    def step(lists):
        want = 0
        for o, m in enumerate(models):  # the owner walks rank 0's segment, then rank 1's, each in list order
            for lst in lists:
                want += sum(m.erase(key) for key in lst if (key >> 63) == o)
        got = each_rank(shards, lambda r: shards[r].drop_hash_array(np.array(lists[r], dtype=np.uint64)))
        assert got == [want, want]
        for s, m in zip(shards, models):
            k, v = s.engine.table.export(0)
            assert list(zip(k.tolist(), v.tolist())) == m.export()
            assert s.engine.table.capacity == cap
        d = {**models[0].items(), **models[1].items()}
        check_against(shards, d)
        q = [key for lst in lists for key in lst] + probes[:20]
        assert each_rank(shards, lambda r: shards[r].get_hash_array(q))[0].tolist() == [d.get(key, 0) for key in q]

    (w0, r0), (w1, r1) = runs
    step([[models[0].slots[cap - 1][0]], [models[1].slots[2][0]]])  # before the wrap; inside the wrapped run
    step([[w1[0], probes[0]], [r0[0]]])  # a key of the other owner and an absent one; a run's first key
    step([r0[100:160:3] + r1[400:420], r1[700:720] + [w0[3]]])
    shards[1].engine.table.set_hash(TOP, 7)  # 2^64-1, listed by both ranks in one call: removed once
    models[1].set(TOP, 7)
    step([[TOP, 0], [TOP]])
    step([[TOP], []])  # absent now
    # drop(kmer) and drop_hash: the k-mer's hash placed in its owner's table first
    kmer = "ACGTTGCAAGGCTTACCGTAG"
    h = int(shards[0].engine.table.hash_windows(kmer.encode())[0])
    shards[h >> 63].engine.table.set_hash(h, 3)
    models[h >> 63].set(h, 3)
    want = models[h >> 63].erase(h) + models[1].erase(r1[5])
    assert want == 2
    each_rank(shards, lambda r: shards[0].drop(kmer) if r == 0 else shards[1].drop_hash(r1[5]))
    for s, m in zip(shards, models):
        k, v = s.engine.table.export(0)
        assert list(zip(k.tolist(), v.tolist())) == m.export()
    with pytest.raises(ValueError, match="kmer size does not match count table ksize"):
        shards[0].drop("ACGT")  # refused before the exchange: no rank is left waiting
    for s in shards:
        s.close()


def test_lists_on_wrapped_and_long_runs(capi):
    """a list (mark and rebuild) across the wrap and an 800-key run, with duplicates from both
    ranks, absent keys homed in the runs and 2^64-1; the capacity stays"""
    shards, models, runs, probes = crafted_shards(capi, 81)
    cap = models[0].cap
    shards[1].engine.table.set_hash(TOP, 9)
    models[1].set(TOP, 9)
    d = {**models[0].items(), **models[1].items()}
    (w0, r0), (w1, r1) = runs
    gone = w0[::2] + r0[::3] + w1[1::2] + r1[::4]
    lists = [gone[: len(gone) // 2] + probes[:40] + [TOP] + gone[-30:], gone[len(gone) // 2:] + gone[:30] + probes[40:] + [TOP]]
    assert sum(map(len, lists)) >= 256
    # Which path ran: an in-place call and a list call of one round each queue the same kernels,
    # but for the erase kernel itself, until each owner that marked keys rebuilds its table once
    # (init_slots_kernel + erase_rebuild_kernel).  Two calls first bring the shards to round 2,
    # from which on every round also waits for its parity buffers.
    for _ in range(2):
        assert dropped_with_launches(shards, [[probes[0]], []])[0] == [0, 0]
    got, in_place = dropped_with_launches(shards, [[probes[1]], [probes[2]]])
    assert got == [0, 0]
    launches = []
    assert drop_and_check(shards, lists, d, launches) == len(gone) + 1
    assert launches == [in_place + 2 * len(shards)]  # both owners marked keys: two rebuilds
    for s in shards:
        assert s.engine.table.capacity == cap
        s.close()


# ---- 4. erase rounds among the other kinds ----------------------------------------------------

def test_erase_between_consume_lookup_and_merge(capi):
    """consume -> erase -> lookup -> merge -> erase -> consume of the same reads, against the model:
    erase rounds keep the round parity of the other kinds"""
    world, k = 2, 21
    bases, offs = reads(5, 12_000)
    counts = oracle_dict(k, bases, offs)
    d = dict(counts)
    shards = consumed_shards(capi, world, k, bases, offs)
    devs = devices_for(capi, world)
    Q = shards[0].engine.info()["round_windows"]
    keys = np.array(sorted(d), dtype=np.uint64)
    rng = np.random.default_rng(4)
    dropped = drop_and_check(shards, [make_list(rng, keys, Q + 7), make_list(rng, keys, 300)], d)
    assert dropped > 0
    q = [keys[r::5] for r in range(world)]
    got = each_rank(shards, lambda r: shards[r].get_hash_array(q[r]))
    for a, b in zip(q, got):
        assert b.tolist() == [d.get(int(h), 0) for h in a.tolist()]
    srcs = []
    for r in range(world):  # (made before the ranks start: allocations synchronise the device)
        t = capi.Table(k, devs[r])
        sk = np.unique(np.concatenate([keys[r::7], rng.integers(0, TOP, 1000, dtype=np.uint64)]))  # dropped keys come back
        t.add_pairs(sk, np.full(len(sk), 2 + r, dtype=np.uint64))
        srcs.append(t)
        for h in sk.tolist():
            d[h] = d.get(h, 0) + 2 + r
    each_rank(shards, lambda r: shards[r].add(srcs[r]))
    check_against(shards, d)
    drop_and_check(shards, [keys[:40], keys[-40:]], d)  # in place
    consume_again(shards, bases, offs)
    for h, c in counts.items():
        d[h] = d.get(h, 0) + c
    check_against(shards, d)
    for t in srcs:
        t.close()
    for s in shards:
        s.close()


# ---- 5. device lists ----------------------------------------------------------------------------

def test_drop_device_lists(capi):
    world, k = 2, 21
    bases, offs = reads(19, 12_000)
    d = oracle_dict(k, bases, offs)
    shards = consumed_shards(capi, world, k, bases, offs)
    devs = devices_for(capi, world)
    Q = shards[0].engine.info()["round_windows"]
    keys = np.array(sorted(d), dtype=np.uint64)
    rng = np.random.default_rng(3)
    lists = [make_list(rng, keys, 2 * Q + 9), make_list(rng, keys, Q // 3)]
    bufs = []
    for r in range(world):
        p = capi.device_alloc(len(lists[r]) * 8, devs[r])
        capi.h2d(p, lists[r], devs[r])
        bufs.append(p)
    want = model_drop(d, lists)
    got = each_rank(shards, lambda r: shards[r].engine.erase_hashes_device(bufs[r], len(lists[r])))
    assert got == [want, want]
    check_against(shards, d)
    for r, p in enumerate(bufs):
        back = np.zeros(len(lists[r]), dtype=np.uint64)
        capi.d2h(back, p, devs[r])
        capi.device_free(p, devs[r])
        assert np.array_equal(back, lists[r])  # the list is left as it was
    for s in shards:
        s.close()


# ---- 6. cuts ------------------------------------------------------------------------------------

def test_cuts_vs_oracle(capi):
    world, k = 2, 21
    bases, offs = reads(23, 12_000)
    truth = OracleTable(k)
    truth.consume_batch(bases, offs, True, nthreads=4)
    shards = consumed_shards(capi, world, k, bases, offs)
    shards[world - 1].engine.table.set_hash(TOP, 3)
    truth.set_hash(TOP, 3)
    shards[0].engine.table.set_hash(5, 0)  # a key held with count 0 (rank 0 owns small keys)
    truth.set_hash(5, 0)
    mx = truth.max
    for kind, m in (("max", mx + 1), ("max", mx), ("min", 0), ("min", 1), ("min", 2), ("max", 2)):
        want = truth.mincut(m) if kind == "min" else truth.maxcut(m)
        got = each_rank(shards, lambda r: shards[r].mincut(m) if kind == "min" else shards[r].maxcut(m))
        assert got == [want, want], (kind, m, got, want)
        tk, tv = truth.items_sorted()
        d = dict(zip(tk.tolist(), tv.tolist()))
        if truth.contains(TOP):
            d[TOP] = truth.get_hash(TOP)
        check_against(shards, d)
    assert TOP not in d and len(d) > 0
    for s in shards:
        s.close()


# ---- 7. two processes -----------------------------------------------------------------------------

def ipc_lists(rank, hashes_of):
    rng = np.random.default_rng(60 + rank)
    present = hashes_of(rank)
    absent = rng.integers(0, TOP, 5000, dtype=np.uint64, endpoint=True)
    q = np.concatenate([present, absent, np.array([0, TOP], dtype=np.uint64), present[:100]])
    rng.shuffle(q)
    return q


def _erase_worker(rank, world, k, conns, out_dir):
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
    bases = synth_reads(n, L, 120_000, seed=13, n_ppm=500)
    offs = uniform_offsets(n, L)
    t = ShardedTable(k, rank, world, device=dev, exchange=exchange, round_windows=1 << 16)
    lo, hi = split_reads(n, rank, world)
    t.consume_batch(bases, offs[lo:hi + 1])
    if rank == world - 1:
        t.engine.table.set_hash(TOP, 4)
    q = ipc_lists(rank, lambda r: t.engine.table.hash_windows(bases[r * 2000 * L:(r * 2000 + 300) * L]))
    listed = t.drop_hash_array(q)
    single = t.drop_hash(int(q[-1]) if rank == 0 else 12345)
    cut = t.mincut(2)
    k_, v_ = t.local_items_sorted()
    np.savez(os.path.join(out_dir, f"erase{rank}.npz"), q=q, keys=k_, vals=v_, counts=np.array([listed, cut], dtype=np.uint64))
    assert single is None
    exchange(b"done")  # nobody unmaps an exchange area a peer may still be reading
    t.close()


def test_drops_in_separate_processes_over_cuda_ipc(capi, tmp_path):
    import multiprocessing as mp

    from oxli_b200.sharded import owner_of

    world, k = 2, 31
    ctx = mp.get_context("spawn")
    a, b = ctx.Pipe()
    procs = [ctx.Process(target=_erase_worker, args=(0, world, k, [a], str(tmp_path))),
             ctx.Process(target=_erase_worker, args=(1, world, k, b, str(tmp_path)))]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    n = 20_000
    truth = OracleTable(k)
    truth.consume_batch(synth_reads(n, L, 120_000, seed=13, n_ppm=500), uniform_offsets(n, L), True, nthreads=4)
    truth.set_hash(TOP, 4)
    parts = [np.load(tmp_path / f"erase{r}.npz") for r in range(world)]
    tk, tv = truth.items_sorted()
    d = dict(zip(tk.tolist(), tv.tolist()))
    d[TOP] = 4
    listed = model_drop(d, [p["q"] for p in parts])
    assert listed > 10_000
    model_drop(d, [[parts[0]["q"][-1]], [12345]])
    cut = 0
    for h in [h for h, c in d.items() if c < 2]:
        del d[h]
        cut += 1
    keys = np.array(sorted(d), dtype=np.uint64)
    vals = np.array([d[int(h)] for h in keys], dtype=np.uint64)
    own = owner_of(keys, world)
    for r, p in enumerate(parts):
        assert p["counts"].tolist() == [listed, cut]
        assert np.array_equal(p["keys"], keys[own == r]) and np.array_equal(p["vals"], vals[own == r])


# ---- 8. refusals ------------------------------------------------------------------------------------

def test_refused_calls_start_no_exchange(capi):
    from oxli_b200.sharded import ShardedTable

    err_invalid = capi.ERR_INVALID
    lib = capi.lib
    h = np.array([5, 9, 7, TOP], dtype=np.uint64)
    n = capi.u64()
    s = capi.Shard(21, 0, 1)
    s.table.count_hashes([5, 5, 9])
    assert lib.oxg_shard_erase_hashes(s._h, None, 4, n) == err_invalid
    assert lib.oxg_shard_erase_hashes_device(s._h, None, 4, n) == err_invalid
    assert lib.oxg_shard_erase_hashes_device(s._h, h.ctypes.data, 4, n) == err_invalid  # a host list
    assert lib.oxg_shard_cut(s._h, 2, 1, n) == err_invalid
    assert s.table.export(1)[0].tolist() == [5, 9]
    assert s.erase_hashes(h[:0]) == 0
    assert s.erase_hashes(h) == 2 and len(s.table) == 0
    s.close()
    # a shard whose peers are not connected: refused at once
    lone = capi.Shard(21, 0, 2)
    assert lib.oxg_shard_erase_hashes(lone._h, h.ctypes.data, 4, n) == err_invalid
    assert b"not connected" in lib.oxg_last_error()
    assert lib.oxg_shard_cut(lone._h, 0, 2, n) == err_invalid
    lone.close()
    # a refused call on one rank of a connected pair returns at once: had it started an exchange,
    # it would have waited for the other rank; both ranks then erase together as usual
    pair = ShardedTable.local(21, 2, devices_for(capi, 2))
    pair[0].engine.table.count_hashes([5, 5, 9])
    pair[1].engine.table.set_hash(TOP, 3)
    for call in (lambda: lib.oxg_shard_erase_hashes(pair[0].engine._h, None, 4, n),
                 lambda: lib.oxg_shard_erase_hashes_device(pair[0].engine._h, h.ctypes.data, 4, n),
                 lambda: lib.oxg_shard_cut(pair[0].engine._h, 7, 1, n)):
        t0 = time.monotonic()
        assert call() == err_invalid
        assert time.monotonic() - t0 < 5
    assert pair[0].local_items_sorted()[0].tolist() == [5, 9] and pair[1].local_items_sorted()[0].tolist() == [TOP]
    got = each_rank(pair, lambda r: pair[r].drop_hash_array([h, np.array([TOP, 5], dtype=np.uint64)][r]))
    assert got == [3, 3]
    assert each_rank(pair, lambda r: len(pair[r])) == [0, 0]
    for p in pair:
        p.close()
