"""The capacity a single table reaches under the growth policy: sketch pre-sizing and the rate
reservation of the partitioned pipeline, the look-ahead of host batches streamed in chunks, the
deferral list and replay of a long hash list, and the rebuild of erase and cut.  The slot counts
are pinned, so that a change to how the host sizes tables shows up here.  Three host chunks of
C3-shaped reads make 22 M keys, and a second pass over them takes the table to 2 GiB; only the
rate reservation asks how much device memory is free, and there the tables are 1 GiB at most, far
below half of a 180 GB card."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

K, L, N_READS, GENOME = 21, 150, 900_000, 2_000_000   # 135 MB of bases: three 64 MiB host chunks
KEMPTY = (1 << 64) - 1

# (capacity, len, counted) after each step
EXPECTED = {
    "device": (67108864, 22335732, 114566917),          # 1 GiB
    "device_again": (134217728, 22335732, 114566917),   # 2 GiB
    "pageable_fresh": (67108864, 22335732, 114566917),
    "hash_list": (16777216, 9991048, 70000000),
}


@pytest.fixture(scope="module")
def capi():
    from oxli_b200 import _capi

    assert _capi.lib.oxg_device_count() > 0, "GPU tests need a CUDA device"
    return _capi


def run_trace(capi) -> dict:
    """Every step's (capacity, len, counted)."""
    out = {}
    tb = N_READS * L
    offs = np.arange(N_READS + 1, dtype=np.uint64) * np.uint64(L)
    d_bases, d_offs = capi.device_alloc(tb + 64), capi.device_alloc(offs.nbytes)
    try:
        # C3-shaped reads: 1 % substitutions, 0.1 % N
        capi.synth_reads_device(d_bases, N_READS, L, GENOME, seed=0xC30001, sub_ppm=10_000, n_ppm=1_000)
        capi.h2d(d_offs, offs)
        t = capi.Table(K)
        for step in ("device", "device_again"):
            st, total, _, _ = t.consume_batch_device(d_bases, d_offs, N_READS, tb, True)
            assert st == 0
            out[step] = (t.capacity, len(t), total)
        t.close()
        bases = np.empty(tb, dtype=np.uint8)
        capi.d2h(bases, d_bases)
    finally:
        capi.device_free(d_bases)
        capi.device_free(d_offs)
    t = capi.Table(K)
    st, total, _, _ = t.consume_batch(bases, offs, True)
    assert st == 0
    out["pageable_fresh"] = (t.capacity, len(t), total)
    t.close()
    del bases
    # 70 M hashes over 10 M distinct keys (two launches), into a table of 1024 slots
    rng = np.random.default_rng(5)
    pool = rng.integers(1, KEMPTY, size=10_000_000, dtype=np.uint64)
    hashes = pool[rng.integers(0, len(pool), size=70_000_000)]
    d_h = capi.device_alloc(hashes.nbytes)
    try:
        capi.h2d(d_h, hashes)
        t = capi.Table(K)
        assert t.capacity == 1024
        total = t.count_hashes_device(d_h, len(hashes))
        out["hash_list"] = (t.capacity, len(t), total)
        t.close()
    finally:
        capi.device_free(d_h)
    return out


@pytest.fixture(scope="module")
def trace(capi):
    return run_trace(capi)


@pytest.mark.parametrize("step", list(EXPECTED))
def test_capacity_trace(trace, step):
    assert trace[step] == EXPECTED[step]


def test_erase_list_then_cut_keeps_capacity(capi):
    """erase_hashes of a list (the rebuild path) and cut rebuild into an array of the same size;
    the out-of-band key 2^64-1 follows each call's own rule."""
    rng = np.random.default_rng(9)
    keys = np.unique(rng.integers(1, KEMPTY, size=300_000, dtype=np.uint64))
    vals = rng.integers(1, 40, size=len(keys), dtype=np.uint64)
    keys = np.append(keys, np.uint64(KEMPTY))
    vals = np.append(vals, np.uint64(7))
    t = capi.Table(K)
    t.add_pairs(keys, vals)
    cap = t.capacity
    want = dict(zip(keys.tolist(), vals.tolist()))

    def same():
        gk, gv = t.export(1)
        wk = np.array(sorted(want), dtype=np.uint64)
        assert np.array_equal(gk, wk)
        assert np.array_equal(gv, np.array([want[x] for x in wk.tolist()], dtype=np.uint64))

    same()
    doomed = np.concatenate([rng.choice(keys[:-1], size=5000, replace=False),
                             rng.integers(1, KEMPTY, size=500, dtype=np.uint64),   # (absent)
                             np.array([KEMPTY], dtype=np.uint64)])
    gone = {x for x in doomed.tolist() if x in want}
    for x in gone:
        del want[x]
    assert t.erase_hashes(doomed) == len(gone)
    assert t.capacity == cap and len(t) == len(want)
    same()
    # the out-of-band key again, below the threshold of the cut
    t.add_pairs(np.array([KEMPTY], dtype=np.uint64), np.array([3], dtype=np.uint64))
    want[KEMPTY] = 3
    low = {x for x, v in want.items() if v < 10}
    for x in low:
        del want[x]
    assert t.cut(0, 10) == len(low)
    assert t.capacity == cap and len(t) == len(want)
    same()
    high = {x for x, v in want.items() if v > 30}
    for x in high:
        del want[x]
    assert t.cut(1, 30) == len(high)
    assert t.capacity == cap and len(t) == len(want)
    same()
    t.close()


if __name__ == "__main__":
    from oxli_b200 import _capi

    for name, got in run_trace(_capi).items():
        print(f"    {name!r}: {got},", flush=True)
