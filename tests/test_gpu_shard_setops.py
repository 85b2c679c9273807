"""Set operations and cosine of two hash-sharded tables (oxg_shard_setop_export, oxg_shard_cosine;
ShardedTable.union / intersection / difference / symmetric_difference / cosine, src/lib.rs:610-655,
727-765) against plain tables holding the same pairs.

A key of A owned by rank r can only be in B's shard on rank r, so each rank computes its own part,
sorted, and the parts in rank order are the whole result sorted.  The model of each result is
np.sort of the plain `_capi.Table.setop` of plain tables built from the same pairs.  As in
test_gpu_shard_dump.py, several shards on one GPU run the same code as one shard per GPU."""
import ctypes
import threading
import time
from decimal import Decimal, localcontext

import numpy as np
import pytest

from synth import synth_reads, uniform_offsets

pytestmark = pytest.mark.gpu
TOP = (1 << 64) - 1
L, G = 150, 150_000
OPS = ("union", "intersection", "difference", "symmetric_difference")


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


def _raised(fn):
    try:
        fn()
    except Exception as e:  # noqa: BLE001
        return e
    return None


def close_all(*groups):
    for g in groups:
        for s in g:
            s.close()


# ---- tables and models ------------------------------------------------------------------------

def fresh(capi, world, k=21):
    from oxli_b200.sharded import ShardedTable

    return ShardedTable.local(k, world, devices_for(capi, world), round_windows=1 << 16)


def consume_reads(shards, bases, offs, lo, hi):
    """reads [lo, hi) of the set, split among the ranks"""
    from oxli_b200.sharded import split_reads

    world = len(shards)

    def consume(r):
        a, b = split_reads(hi - lo, r, world)
        shards[r].consume_batch(bases, offs[lo + a:lo + b + 1])

    run_ranks([lambda r=r: consume(r) for r in range(world)])


def half_overlapping(capi, world, k, seed, n=18_000):
    """A counts reads [0, 2n/3), B reads [n/3, n): they share half of each one's reads"""
    bases = synth_reads(n, L, G, seed=seed, sub_ppm=5000, n_ppm=800)
    offs = uniform_offsets(n, L)
    A, B = fresh(capi, world, k), fresh(capi, world, k)
    consume_reads(A, bases, offs, 0, 2 * n // 3)
    consume_reads(B, bases, offs, n // 3, n)
    return A, B


def with_pairs(capi, world, keys, vals, k=21):
    """fresh shards holding these (key, count) pairs: rank 0 adds a plain table of all of them"""
    shards = fresh(capi, world, k)
    devs = devices_for(capi, world)
    srcs = [capi.Table(k, devs[r]) for r in range(world)]
    if len(keys):
        srcs[0].add_pairs(np.asarray(keys, dtype=np.uint64), np.asarray(vals, dtype=np.uint64))
    each_rank(shards, lambda r: shards[r].add(srcs[r]))
    for t in srcs:
        t.close()
    return shards


def pairs_of(shards):
    """every rank's pairs (plain-table export of its shard, not the code under test)"""
    parts = [s.engine.table.export(0) for s in shards]
    return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])


def plain_of(capi, shards, k):
    t = capi.Table(k, 0)
    keys, vals = pairs_of(shards)
    if len(keys):
        t.add_pairs(keys, vals)
    assert len(t) == len(keys)
    return t


def ascending(a):
    return bool((a[1:] > a[:-1]).all())


def assemble(parts, world):
    """the whole result from every rank's (keys, start, total), checking how the parts fit"""
    from oxli_b200.sharded import owner_of

    total = parts[0][2]
    before = 0
    for r, (keys, start, tot) in enumerate(parts):
        assert tot == total and start == before, (r, start, before, tot, total)
        assert ascending(keys), r
        assert (owner_of(keys, world) == r).all(), r
        before += len(keys)
    assert before == total
    return np.concatenate([p[0] for p in parts]) if parts else np.zeros(0, dtype=np.uint64)


def check_setops(capi, A, B, k):
    """every op of A with B against np.sort of the plain tables' setop; returns the wholes"""
    world = len(A)
    pa, pb = plain_of(capi, A, k), plain_of(capi, B, k)
    inter, uni = each_rank(A, lambda r: A[r].setop_sizes(B[r]))[0]
    out = {}
    for op, name in enumerate(OPS):
        parts = each_rank(A, lambda r: getattr(A[r], name)(B[r]))
        whole = assemble(parts, world)
        want = np.sort(pa.setop(pb, op))
        assert whole.dtype == np.uint64 and np.array_equal(whole, want), name
        out[name] = whole
    assert len(out["intersection"]) == inter and len(out["union"]) == uni
    pa.close()
    pb.close()
    return out


# ---- 1. consumed tables ---------------------------------------------------------------------------

@pytest.mark.parametrize("world, k", [(1, 21), (2, 21), (4, 21), (2, 31)])
def test_setops_vs_plain_tables(capi, world, k):
    A, B = half_overlapping(capi, world, k, seed=60 + world + k)
    got = check_setops(capi, A, B, k)
    assert 0 < len(got["intersection"]) < len(got["union"])
    assert len(got["difference"]) > 0 and len(got["symmetric_difference"]) > len(got["difference"])
    close_all(A, B)


# ---- 2. crafted tables ------------------------------------------------------------------------------

def owned_keys(rng, world, ranks, n):
    """n distinct random keys (never 2^64-1) owned by the given ranks"""
    shift = 64 - (world.bit_length() - 1)
    per = [rng.integers(0, 1 << shift, n, dtype=np.uint64) | (np.uint64(r) << np.uint64(shift)) if world > 1
           else rng.integers(0, TOP, n, dtype=np.uint64) for r in ranks]
    keys = np.unique(np.concatenate(per))
    return keys[keys != TOP]


@pytest.mark.parametrize("where", ["a_only", "b_only", "both", "neither"])
def test_top_key_zero_counts_and_an_empty_rank(capi, where):
    """2^64-1 in A, B, both or neither; keys held with count 0 (members); rank 1 owns nothing"""
    world = 4
    rng = np.random.default_rng(7)
    keys = owned_keys(rng, world, (0, 2, 3), 3000)
    ka, kb = keys[: 2000], keys[1000:]
    va = rng.integers(0, 3, len(ka), dtype=np.uint64)  # a third held with count 0
    vb = rng.integers(0, 3, len(kb), dtype=np.uint64)
    if where in ("a_only", "both"):
        ka, va = np.append(ka, np.uint64(TOP)), np.append(va, np.uint64(0))
    if where in ("b_only", "both"):
        kb, vb = np.append(kb, np.uint64(TOP)), np.append(vb, np.uint64(5))
    A, B = with_pairs(capi, world, ka, va), with_pairs(capi, world, kb, vb)
    assert len(A[1].engine.table) == 0 and len(B[1].engine.table) == 0
    got = check_setops(capi, A, B, 21)
    sa, sb = where in ("a_only", "both"), where in ("b_only", "both")
    want_top = {"union": sa or sb, "intersection": sa and sb, "difference": sa and not sb, "symmetric_difference": sa != sb}
    for name, whole in got.items():
        assert (len(whole) > 0 and whole[-1] == TOP) == want_top[name], name
    close_all(A, B)


@pytest.mark.parametrize("world", [1, 2])
def test_empty_tables(capi, world):
    A, B = fresh(capi, world), fresh(capi, world)
    for name in OPS:
        for keys, start, total in each_rank(A, lambda r: getattr(A[r], name)(B[r])):
            assert len(keys) == 0 and start == 0 and total == 0
    assert each_rank(A, lambda r: A[r].cosine(B[r])) == [0.0] * world
    rng = np.random.default_rng(3)
    keys = owned_keys(rng, world, range(world), 500)
    C = with_pairs(capi, world, keys, np.ones(len(keys), dtype=np.uint64))
    check_setops(capi, C, A, 21)
    check_setops(capi, A, C, 21)
    assert each_rank(A, lambda r: C[r].cosine(A[r])) == [0.0] * world
    assert each_rank(A, lambda r: A[r].cosine(C[r])) == [0.0] * world
    close_all(A, B, C)


def test_a_table_with_itself(capi):
    world = 2
    rng = np.random.default_rng(9)
    keys = np.append(owned_keys(rng, world, (0, 1), 4000), np.uint64(TOP))
    A = with_pairs(capi, world, keys, rng.integers(0, 4, len(keys), dtype=np.uint64))
    want = np.sort(keys)
    for name in OPS:
        whole = assemble(each_rank(A, lambda r: getattr(A[r], name)(A[r])), world)
        assert np.array_equal(whole, want if name in ("union", "intersection") else want[:0]), name
    close_all(A)


def test_a_part_larger_than_the_bounce_buffer(capi):
    """rank 0's union holds 9 M keys (72 MB: two pieces through the 64 MiB staging chunk, the last
    one partial) over many radix tiles; rank 1 owns nothing"""
    world = 2
    rng = np.random.default_rng(21)
    keys = np.unique(rng.integers(0, 1 << 63, 9_300_000, dtype=np.uint64))[:9_000_000]
    perm = rng.permutation(len(keys))
    ka, kb = keys[perm[:6_000_000]], keys[perm[3_000_000:]]
    A = with_pairs(capi, world, ka, np.ones(len(ka), dtype=np.uint64))
    B = with_pairs(capi, world, kb, np.full(len(kb), 2, dtype=np.uint64))
    want = {"union": keys, "intersection": np.intersect1d(ka, kb), "difference": np.setdiff1d(ka, kb),
            "symmetric_difference": np.setxor1d(ka, kb)}
    for name in OPS:
        parts = each_rank(A, lambda r: getattr(A[r], name)(B[r]))
        assert len(parts[1][0]) == 0
        assert np.array_equal(assemble(parts, world), want[name]), name
    assert len(want["union"]) * 8 > 64 << 20  # (the shard's staging chunk: 64 MiB by default)
    close_all(A, B)


# ---- 3. cosine ------------------------------------------------------------------------------------------

def exact_cosine(ka, va, kb, vb):
    """cosine of two count tables from Python integers, evaluated at 40 digits"""
    a = dict(zip(np.asarray(ka).tolist(), np.asarray(va).tolist()))
    b = dict(zip(np.asarray(kb).tolist(), np.asarray(vb).tolist()))
    dot = sum(c * b[key] for key, c in a.items() if key in b)
    sa, sb = sum(c * c for c in a.values()), sum(c * c for c in b.values())
    with localcontext() as ctx:
        ctx.prec = 40
        return dot, Decimal(dot) / (Decimal(sa) * Decimal(sb)).sqrt()


def assert_cosine(got, want, n_a, n_b):
    # the squares are summed in doubles in any order: each sum is off by at most (n - 1) rounding
    # steps, the rest (the squares, the square roots, the product, dot's conversion and the
    # quotient) adds a few more
    bound = (n_a + n_b + 4) * 2.0 ** -53
    assert abs(Decimal(got) - want) <= Decimal(bound) * want, (got, want)


@pytest.mark.parametrize("world", [1, 2, 4])
def test_cosine_exact_with_large_counts_and_side_entries(capi, world):
    rng = np.random.default_rng(30 + world)
    keys = rng.permutation(owned_keys(rng, world, range(world), 6000))
    shared, a_only, b_only = keys[:2000], keys[2000:4000], keys[4000:]
    # counts up to 2^31 - 1, the dot product kept below 2^64 (the reference sums it in u64; how a
    # wrapped sum behaves is not something a 40-digit value can stand in for)
    top = np.uint64((1 << 31) - 1)
    va_s = rng.integers(0, 1 << 20, len(shared), dtype=np.uint64)
    vb_s = rng.integers(0, 1 << 20, len(shared), dtype=np.uint64)
    va_s[:2] = top
    vb_s[:2] = top
    ka = np.concatenate([shared, a_only])
    va = np.concatenate([va_s, rng.integers(0, 1 << 31, len(a_only), dtype=np.uint64)])
    kb = np.concatenate([shared, b_only])
    vb = np.concatenate([vb_s, rng.integers(0, 1 << 31, len(b_only), dtype=np.uint64)])
    ka, va = np.append(ka, np.uint64(TOP)), np.append(va, np.uint64((1 << 31) - 1))  # side entries count
    kb, vb = np.append(kb, np.uint64(TOP)), np.append(vb, np.uint64(1 << 30))
    dot, want = exact_cosine(ka, va, kb, vb)
    assert dot < 1 << 64  # (no wrap-around: the exact value is the reference's)
    A, B = with_pairs(capi, world, ka, va), with_pairs(capi, world, kb, vb)
    got = each_rank(A, lambda r: A[r].cosine(B[r]))
    assert all(g == got[0] for g in got)  # the same double on every rank
    assert_cosine(got[0], want, len(ka), len(kb))
    pa, pb = plain_of(capi, A, 21), plain_of(capi, B, 21)
    assert_cosine(pa.cosine(pb), want, len(ka), len(kb))
    # without the side entries the value moves: they are counted
    _, without = exact_cosine(ka[:-1], va[:-1], kb[:-1], vb[:-1])
    assert abs(Decimal(got[0]) - without) > Decimal(1e-12) * without
    pa.close()
    pb.close()
    close_all(A, B)


def test_cosine_of_zero_counts_is_zero(capi):
    world = 2
    rng = np.random.default_rng(5)
    keys = owned_keys(rng, world, (0, 1), 1000)
    A = with_pairs(capi, world, keys, np.zeros(len(keys), dtype=np.uint64))
    B = with_pairs(capi, world, keys[::2], np.full(len(keys[::2]), 3, dtype=np.uint64))
    for x, y in ((A, B), (B, A), (A, A)):
        assert each_rank(A, lambda r: x[r].cosine(y[r])) == [0.0] * world
    close_all(A, B)


# ---- 4. refusals, disagreements, failures ---------------------------------------------------------------

def test_refusals_start_no_exchange_and_change_nothing(capi):
    lib, err_invalid = capi.lib, capi.ERR_INVALID
    A, B = half_overlapping(capi, 2, 21, seed=4, n=3000)
    one = fresh(capi, 1)
    lone = capi.Shard(21, 0, 2)  # a shard whose peers are not connected
    before = [each_rank(A, lambda r: A[r].digest()), each_rank(B, lambda r: B[r].digest())]
    live = lib.oxg_live_allocations()
    n, s, t, d = capi.u64(), capi.u64(), capi.u64(), ctypes.c_double()
    buf = np.zeros(8, dtype=np.uint64)
    for r in range(2):
        a, b = A[r].engine._h, B[r].engine._h
        other = B[1 - r].engine._h  # same n_ranks, another rank
        calls = [lambda: lib.oxg_shard_setop_export(None, b, 0, None, 0, n, s, t),
                 lambda: lib.oxg_shard_setop_export(a, None, 0, None, 0, n, s, t),
                 lambda: lib.oxg_shard_setop_export(lone._h, b, 0, None, 0, n, s, t),
                 lambda: lib.oxg_shard_setop_export(a, lone._h, 0, None, 0, n, s, t),
                 lambda: lib.oxg_shard_setop_export(a, b, 0, None, 0, None, s, t),
                 lambda: lib.oxg_shard_setop_export(a, b, 0, None, 4, n, s, t),
                 lambda: lib.oxg_shard_setop_export(a, b, 4, buf.ctypes.data, 8, n, s, t),
                 lambda: lib.oxg_shard_setop_export(a, b, -1, buf.ctypes.data, 8, n, s, t),
                 lambda: lib.oxg_shard_setop_export(a, other, 1, buf.ctypes.data, 8, n, s, t),
                 lambda: lib.oxg_shard_setop_export(a, one[0].engine._h, 1, buf.ctypes.data, 8, n, s, t),
                 lambda: lib.oxg_shard_cosine(None, b, d),
                 lambda: lib.oxg_shard_cosine(a, None, d),
                 lambda: lib.oxg_shard_cosine(lone._h, b, d),
                 lambda: lib.oxg_shard_cosine(a, b, None),
                 lambda: lib.oxg_shard_cosine(a, other, d),
                 lambda: lib.oxg_shard_cosine(one[0].engine._h, b, d)]
        for i, call in enumerate(calls):
            t0 = time.monotonic()
            assert call() == err_invalid, (r, i)
            assert time.monotonic() - t0 < 5, (r, i)  # refused on one rank alone: no exchange was started
    if lib.oxg_device_count() > 1:  # shards of one rank on two devices
        from oxli_b200.sharded import ShardedTable

        X, Y = ShardedTable.local(21, 1, [0]), ShardedTable.local(21, 1, [1])
        assert lib.oxg_shard_setop_export(X[0].engine._h, Y[0].engine._h, 0, None, 0, n, s, t) == err_invalid
        assert lib.oxg_shard_cosine(X[0].engine._h, Y[0].engine._h, d) == err_invalid
        close_all(X, Y)
    assert lib.oxg_live_allocations() == live
    assert [each_rank(A, lambda r: A[r].digest()), each_rank(B, lambda r: B[r].digest())] == before
    with pytest.raises(TypeError):
        A[0].union(B[0].engine)
    check_setops(capi, A, B, 21)  # both tables as usable as before
    lone.close()
    close_all(A, B, one)


def test_ranks_that_pass_different_ops_all_get_valueerror(capi):
    A, B = half_overlapping(capi, 2, 21, seed=8, n=3000)
    errs = each_rank(A, lambda r: _raised(lambda: getattr(A[r], OPS[r])(B[r])))
    for r, e in enumerate(errs):
        assert isinstance(e, ValueError) and "different set operations" in str(e), (r, e)
    check_setops(capi, A, B, 21)
    close_all(A, B)


def test_an_allocation_failure_on_one_rank_reaches_every_rank_promptly(capi):
    lib = capi.lib
    A, B = half_overlapping(capi, 2, 21, seed=11, n=6000)
    first = assemble(each_rank(A, lambda r: A[r].union(B[r])), 2)
    live = lib.oxg_live_allocations()
    lib.oxg_fail_allocation_after(1)  # the first reservation, on whichever rank makes it first
    try:
        t0 = time.monotonic()
        errs = each_rank(A, lambda r: _raised(lambda: A[r].union(B[r])))
        took = time.monotonic() - t0
    finally:
        left = lib.oxg_fail_allocation_after(0)
    assert left == 0
    assert took < 10, took  # far inside the 30 s a peer waits before it gives up
    for r, e in enumerate(errs):
        assert isinstance(e, MemoryError), (r, e)
    assert lib.oxg_live_allocations() == live
    assert np.array_equal(assemble(each_rank(A, lambda r: A[r].union(B[r])), 2), first)
    close_all(A, B)


# ---- 5. among the other calls ------------------------------------------------------------------------------

def test_setops_see_consume_erase_and_plain_adds(capi):
    world, k = 2, 21
    n = 9000
    bases = synth_reads(n, L, G, seed=13, sub_ppm=5000, n_ppm=800)
    offs = uniform_offsets(n, L)
    A, B = fresh(capi, world, k), fresh(capi, world, k)
    consume_reads(A, bases, offs, 0, 3000)
    consume_reads(B, bases, offs, 1500, 4500)
    check_setops(capi, A, B, k)
    consume_reads(A, bases, offs, 4500, 6000)  # after a consume
    check_setops(capi, A, B, k)
    keys, _ = pairs_of(B)
    gone = [keys[::3], keys[1::7]]
    each_rank(B, lambda r: B[r].drop_hash_array(gone[r]))  # after an erase
    check_setops(capi, A, B, k)
    rng = np.random.default_rng(2)
    from oxli_b200.sharded import owner_of

    for r in range(world):  # after plain adds on a shard's own table (keys that rank owns)
        extra = owned_keys(rng, world, (r,), 300)
        assert (owner_of(extra, world) == r).all()
        A[r].engine.table.add_pairs(extra, np.zeros(len(extra), dtype=np.uint64))
    A[world - 1].engine.table.set_hash(TOP, 2)
    got = check_setops(capi, A, B, k)
    assert got["difference"][-1] == TOP
    close_all(A, B)
