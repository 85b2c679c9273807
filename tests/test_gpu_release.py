"""Error returns release what the call allocated: a plain table's and a one-rank shard's life,
with each allocation in turn made to fail as out of memory (oxg_fail_allocation_after), ends
with the library holding as many CUDA buffers, events and streams as a clean run leaves behind
(oxg_live_allocations).  Only one-rank shards: a rank that returns in the middle of a collective
would leave its peers waiting for it."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
K = 21


@pytest.fixture(scope="module")
def capi():
    from oxli_b200 import _capi

    assert _capi.lib.oxg_device_count() > 0, "GPU tests need a CUDA device"
    return _capi


def reads(n_reads, read_len=150, genome_len=100_000, seed=7):
    """reads drawn from a small random genome (few distinct k-mers however many reads)"""
    rng = np.random.default_rng(seed)
    genome = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, genome_len)]
    starts = rng.integers(0, genome_len - read_len, n_reads)
    bases = genome[starts[:, None] + np.arange(read_len)].ravel()
    return np.ascontiguousarray(bases), np.arange(n_reads + 1, dtype=np.uint64) * read_len


def plain_life(capi, made, data):
    bases, offsets = data
    t = capi.Table(K, capacity_hint=200_000)
    made.append(t)
    t.consume_batch(bases, offsets)
    doomed = np.concatenate([t.hash_windows(bases[o:o + 150]) for o in (0, 150, 300)])  # three whole reads
    assert t.erase_hashes(doomed) > 0
    u = capi.Table(K)
    made.append(u)
    u.count_hashes(t.hash_windows(bases[1000:2000]))
    t.setop(u, 0)
    keys, vals = t.export(2)
    assert len(keys) == len(t)


def shard_life(capi, made, data, path):
    bases, offsets = data
    s = capi.Shard(K, 0, 1, capacity_hint=200_000, round_windows=1 << 20)
    made.append(s)
    s.consume_batch(bases, offsets)
    keys = np.concatenate([s.table.hash_windows(bases[o:o + 150]) for o in (0, 150, 300)])  # three whole reads
    assert (s.get_hashes(keys) > 0).all()
    assert s.erase_hashes(keys[:300]) > 0
    p = capi.Table(K)
    made.append(p)
    p.count_hashes(keys)
    s.merge_table(p)
    s.export_pairs(2)
    s.dump(path, 0)


def run(capi, life):
    """life() once; returns its status (OK or the failing call's) and destroys what it made"""
    made = []
    try:
        life(made)
        return capi.OK
    except capi.OxliError as e:
        return e.status
    finally:
        for obj in reversed(made):
            obj.close()


def check_releases(capi, life):
    lib = capi.lib
    assert run(capi, life) == capi.OK
    baseline = lib.oxg_live_allocations()
    n = 0
    while True:
        n += 1
        lib.oxg_fail_allocation_after(n)
        try:
            st = run(capi, life)
        finally:
            left = lib.oxg_fail_allocation_after(0)  # 0: the n-th allocation was made, and failed
        assert st in (capi.OK, capi.ERR_NOMEM), (n, st, lib.oxg_last_error())
        assert (st == capi.OK) == (left > 0), f"allocation {n}: status {st}, countdown left {left}"
        if st == capi.OK:
            break  # the run made fewer than n allocations: every one of them has failed once
    assert n > 10, "too few allocations to be the whole life of a table"
    assert run(capi, life) == capi.OK
    assert lib.oxg_live_allocations() == baseline, n


def test_plain_table_releases_on_every_error_return(capi):
    # a host batch of three staging chunks (64 MiB each by default), its reads from a small genome
    data = reads(1_000_000)
    check_releases(capi, lambda made: plain_life(capi, made, data))


def test_one_rank_shard_releases_on_every_error_return(capi, tmp_path):
    data = reads(50_000)
    path = str(tmp_path / "dump.txt")
    check_releases(capi, lambda made: shard_life(capi, made, data, path))
    assert os.path.getsize(path) > 0
