"""The five routes by which reads enter a table -- oxg_consume_batch from pageable and from pinned
memory, oxg_consume_batch_device, and oxg_shard_consume_batch / oxg_shard_consume_batch_device
with two shards on one GPU -- against the CPU oracle, in both modes, on one ragged batch that spans
several 64 MiB host staging chunks and several shard rounds.  All of them share one error-mode
driver per table kind and one staging ring, so they must agree read for read."""
import threading

import numpy as np
import pytest

from oracle import OracleTable

pytestmark = pytest.mark.gpu
K = 31
WORLD = 2


@pytest.fixture(scope="module")
def capi():
    from oxli_b200 import _capi

    assert _capi.lib.oxg_device_count() > 0, "GPU tests need a CUDA device"
    return _capi


@pytest.fixture(scope="module")
def batch(capi):
    """Reads of 0..300 bases cut from 150 MB of generated sequence, one non-ACGT byte in the
    middle of a read in the second host chunk.  Returns (bases, offsets, bad read, split read)."""
    total = 150_000_000
    d_bases = capi.device_alloc(total + 64)
    try:
        capi.synth_reads_device(d_bases, total // 150, 150, 300_000, seed=13, sub_ppm=500)
        bases = np.empty(total, dtype=np.uint8)
        capi.d2h(bases, d_bases)
    finally:
        capi.device_free(d_bases)
    rng = np.random.default_rng(13)
    lens = rng.integers(0, 301, size=total // 100)
    ends = np.cumsum(lens)
    ends = ends[ends < total]
    offs = np.concatenate([[0], ends, [total]]).astype(np.uint64)
    r_bad = int(np.searchsorted(offs, 100_000_000))            # a read starting in the second chunk
    while int(offs[r_bad + 1]) - int(offs[r_bad]) < 200:
        r_bad += 1
    bases[int(offs[r_bad]) + 100] = ord("N")
    split = r_bad - 1000                                        # rank 1 holds the bad read
    return bases, offs, r_bad, split


@pytest.fixture(scope="module")
def truth(batch):
    """(counted, err_read, err_pos) and the sorted (hash, count) table per mode."""
    bases, offs, r_bad, _ = batch
    out = {}
    for skip in (True, False):
        ora = OracleTable(K)
        res = ora.consume_batch(bases, offs, skip, nthreads=8)
        out[skip] = (res, ora.items_sorted())
    assert out[False][0][1] == r_bad and out[True][0][1] == -1
    return out


def assert_items(got, want):
    assert len(got[0]) == len(want[0])
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


@pytest.mark.parametrize("skip", [True, False])
@pytest.mark.parametrize("route", ["pageable", "pinned", "device"])
def test_one_table(capi, batch, truth, route, skip):
    bases, offs, _, _ = batch
    (want, items) = truth[skip]
    t = capi.Table(K)
    if route == "device":
        d_b, d_o = capi.device_alloc(bases.nbytes + 64), capi.device_alloc(offs.nbytes)
        try:
            capi.h2d(d_b, bases); capi.h2d(d_o, offs)
            st, total, er, ep = t.consume_batch_device(d_b, d_o, len(offs) - 1, bases.nbytes, skip)
        finally:
            capi.device_free(d_b); capi.device_free(d_o)
    else:
        buf = bases
        if route == "pinned":
            buf = capi.pinned_empty(bases.nbytes)
            buf[:] = bases
        st, total, er, ep = t.consume_batch(buf, offs, skip)
        if route == "pinned":
            capi.pinned_free(buf)
    assert st == (capi.OK if skip else capi.ERR_BAD_KMER)
    assert (total, er, ep) == want
    assert_items(t.export(1), items)
    t.close()


def run_ranks(fns):
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


@pytest.mark.parametrize("skip", [True, False])
@pytest.mark.parametrize("route", ["host", "device"])
def test_two_shards(capi, batch, truth, route, skip):
    bases, offs, _, split = batch
    (want, items) = truth[skip]
    n = len(offs) - 1
    parts = [(0, split), (split, n)]
    shards = [capi.Shard(K, r, WORLD, device=0, round_windows=1 << 16) for r in range(WORLD)]
    capi.Shard.connect_local(shards)
    # device buffers exist before the ranks start: an allocation by one rank while the other
    # waits for it inside a kernel on the same GPU would deadlock
    bufs = []
    if route == "device":
        for lo, hi in parts:
            b0, b1 = int(offs[lo]), int(offs[hi])
            d_b, d_o = capi.device_alloc(b1 - b0 + 64), capi.device_alloc((hi - lo + 1) * 8)
            capi.h2d(d_b, bases[b0:b1]); capi.h2d(d_o, offs[lo:hi + 1] - np.uint64(b0))
            bufs.append((d_b, d_o, hi - lo, b1 - b0))
    res = [None] * WORLD

    def rank_fn(r):
        def go():
            lo, hi = parts[r]
            if route == "device":
                res[r] = shards[r].consume_batch_device(*bufs[r], skip)
            else:
                res[r] = shards[r].consume_batch(bases, offs[lo:hi + 1], skip)
        return go

    try:
        run_ranks([rank_fn(r) for r in range(WORLD)])
    finally:
        for d_b, d_o, _, _ in bufs:
            capi.device_free(d_b); capi.device_free(d_o)
    counted, er, ep = want
    assert res[0][0] == capi.OK and res[0][3] == -1
    assert res[1][0] == (capi.OK if skip else capi.ERR_BAD_KMER)
    got_er = -1 if skip else res[1][3] + split
    assert (res[0][1] + res[1][1], got_er, res[1][4]) == (counted, er, ep)
    ks, vs = zip(*[s.table.export(1) for s in shards])
    allk, allv = np.concatenate(ks), np.concatenate(vs)
    order = np.argsort(allk, kind="stable")
    assert_items((allk[order], allv[order]), items)
    for s in shards:
        s.close()


@pytest.mark.parametrize("skip", [True, False])
def test_decreasing_offsets_are_refused(capi, skip):
    # first and last boundary in order, one pair inside out of order.  The shard is N = 1: a rank
    # that fails while its peers wait for it would leave them in the flag wait.
    bases = np.frombuffer(b"ACGT" * 25_000, dtype=np.uint8)
    offs = np.arange(0, 100_001, 100, dtype=np.uint64)
    offs[500], offs[501] = offs[501], offs[500]
    pinned = capi.pinned_empty(bases.nbytes)
    pinned[:] = bases
    try:
        for buf in (bases, pinned):
            with pytest.raises(capi.OxliError) as e:
                capi.Table(K).consume_batch(buf, offs, skip)
            assert e.value.status == capi.ERR_INVALID
    finally:
        capi.pinned_free(pinned)
    shard = capi.Shard(K, 0, 1)
    with pytest.raises(capi.OxliError) as e:
        shard.consume_batch(bases, offs, skip)
    assert e.value.status == capi.ERR_INVALID
    shard.close()
