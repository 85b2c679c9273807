"""Sharded consume into a shard near its load limit, bit for bit against the CPU oracle.

Pass B of an owner reads every rank's fragments, so one round can bring one shard every window
start of every rank: a tandem repeat whose k-mers one rank owns, or a round larger than the
deferral lists were sized for.  Once a shard is at its load limit each such occurrence may become
its own deferral entry.  Every case here fills the shards to about 75 % of a hinted capacity with
batches of one round each (no growth monitor runs for them), asserts that layout, then sends the
burst and compares the whole table with the oracle: keys and counts, counted and absorbed, stats,
histogram, digest, and the owner of every key.  The controls run the same inputs into shards
hinted for the final size."""
import json
import itertools
import os
import sys
import threading

import numpy as np
import pytest

import oracle
from oracle import OracleTable
from oxli_b200.sharded import owner_of
from synth import synth_reads, uniform_offsets

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K, L = 21, 150
WPR = L - K + 1              # windows per read
FILL = 0.755                 # fill before the burst, as a share of capacity
BATCH_WINDOWS = 3 << 20      # windows of one fill batch over all ranks: its worst case fits a shard's 4 Mi deferral list
FAR = 1 << 40                # genome length: reads of it share no k-mer


# ---- input builders (CPU) -------------------------------------------------------------------

def unit_kmers(unit: bytes, k: int = K) -> np.ndarray:
    """The distinct hashes of the k-mers of unit repeated in tandem."""
    return np.unique(oracle.hash_windows(unit * (k // len(unit) + 3), k))


def repeat_unit(world: int, taken: np.ndarray | None = None, k: int = K) -> tuple[bytes, np.ndarray]:
    """The first unit of 4-6 bases, in ACGT order, whose tandem repeat has only k-mers that rank 0
    owns at `world`, none of them among the sorted hashes `taken`."""
    for p in (4, 5, 6):
        for u in itertools.product(b"ACGT", repeat=p):
            h = unit_kmers(bytes(u), k)
            if np.all(owner_of(h, world) == 0) and (taken is None or not np.isin(h, taken).any()):
                return bytes(u), h
    raise AssertionError(f"no repeat unit of 4-6 bases is owned by rank 0 of {world}")


def repeat_reads(unit: bytes, n_reads: int) -> tuple[np.ndarray, np.ndarray]:
    read = (unit * (L // len(unit) + 1))[:L]
    return np.frombuffer(read * n_reads, dtype=np.uint8).copy(), uniform_offsets(n_reads, L)


ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def greedy_reads(n_reads: int, world: int, seed: int, hash_windows, k: int = K) -> tuple[np.ndarray, np.ndarray]:
    """Reads of L bases built base by base: after k - 1 random bases, each next base is, of the four
    tried in a random order, the first whose new k-mer rank 0 owns at `world`, or the first tried
    when none is.  hash_windows(bytes) -> per-window hashes ranks the candidates: the k-mers of all
    reads and bases sit end to end, so every k-th window is one."""
    rng = np.random.default_rng(seed)
    reads = np.empty((n_reads, L), dtype=np.uint8)
    reads[:, :k - 1] = ACGT[rng.integers(0, 4, (n_reads, k - 1))]
    rows = np.arange(n_reads)
    for j in range(k - 1, L):
        order = rng.permuted(np.tile(np.arange(4), (n_reads, 1)), axis=1)
        cand = np.empty((n_reads, 4, k), dtype=np.uint8)
        cand[:, :, :k - 1] = reads[:, None, j - k + 1:j]
        cand[:, :, k - 1] = ACGT[order]
        h = np.asarray(hash_windows(cand.reshape(-1)))[::k].reshape(n_reads, 4)
        own = owner_of(h, world) == 0
        reads[:, j] = ACGT[order[rows, own.argmax(axis=1)]]  # (argmax: the first owned one, else the first)
    return reads.reshape(-1), uniform_offsets(n_reads, L)


def read_hashes(bases: np.ndarray, n_reads: int, k: int = K) -> np.ndarray:
    """oracle hashes of every window inside a read of L bases, one row per read"""
    h = oracle.hash_windows(bases, k)
    at = (np.arange(n_reads)[:, None] * L + np.arange(L - k + 1)[None, :]).reshape(-1)
    return h[at].reshape(n_reads, L - k + 1)


def test_greedy_read_builder():
    world, n = 2, 300
    bases, offs = greedy_reads(n, world, 7, lambda a: oracle.hash_windows(a, K))
    assert len(offs) == n + 1 and len(bases) == n * L
    h = read_hashes(bases, n)
    own = owner_of(h, world) == 0
    assert 0.9 <= own.mean() <= 0.97, own.mean()  # 15/16 when the four candidates are independent
    # where a read's k-mer is not rank 0's, none of the four it could have had is
    for r, i in zip(*np.nonzero(~own)):
        pre = bytes(bases[r * L + i:r * L + i + K - 1])
        alt = [oracle.hash_kmer(pre + bytes([b]), K) for b in b"ACGT"]
        assert np.all(owner_of(np.array(alt, dtype=np.uint64), world) != 0)


@pytest.mark.parametrize("world", [4, 8])
def test_repeat_unit_builder(world):
    unit, h = repeat_unit(world)
    assert 4 <= len(unit) <= 6
    assert np.all(owner_of(h, world) == 0)
    bases, offs = repeat_reads(unit, 3)
    for r in range(3):
        got = np.unique(oracle.hash_windows(bases[int(offs[r]):int(offs[r + 1])], K))
        assert np.array_equal(got, h)
    if world == 4:  # a unit whose k-mers are taken is passed over
        other, h2 = repeat_unit(world, taken=h)
        assert other != unit and not np.isin(h2, h).any() and np.all(owner_of(h2, world) == 0)


# ---- running the ranks ----------------------------------------------------------------------

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


def make_shards(capi, world, hint, round_windows):
    from oxli_b200.sharded import ShardedTable

    n = capi.lib.oxg_device_count()
    return ShardedTable.local(K, world, [r % n for r in range(world)], capacity_hint=hint, round_windows=round_windows)


def consume(capi, shards, parts, device=False):
    """One collective batch: rank r consumes parts[r] = (bases, offsets into bases), from host memory
    or from device buffers made before the ranks start (an allocation while a peer on the same GPU
    waits in a kernel would deadlock).  Returns the sums of counted and absorbed."""
    got = [0] * len(shards)
    bufs = []
    if device:
        for s, (b, o) in zip(shards, parts):
            seg = np.ascontiguousarray(b[int(o[0]):int(o[-1])])
            rel = np.ascontiguousarray(o - o[0], dtype=np.uint64)
            dev = s.engine.device
            d_b, d_o = capi.device_alloc(len(seg) + 64, dev), capi.device_alloc(len(rel) * 8, dev)
            capi.h2d(d_b, seg, dev)
            capi.h2d(d_o, rel, dev)
            bufs.append((d_b, d_o, len(rel) - 1, len(seg)))

    def rank_fn(r):
        def go():
            if device:
                d_b, d_o, n, total = bufs[r]
                got[r] = shards[r].consume_batch_device(d_b, d_o, n, total)
            else:
                got[r] = shards[r].consume_batch(*parts[r])
        return go

    try:
        run_ranks([rank_fn(r) for r in range(len(shards))])
    finally:
        for s, (d_b, d_o, _, _) in zip(shards, bufs):
            capi.device_free(d_b, s.engine.device)
            capi.device_free(d_o, s.engine.device)
    return sum(got), sum(s.last_absorbed for s in shards)


def split(offs, world):
    """every rank's block of the reads of offs"""
    n = len(offs) - 1
    return [offs[n * r // world:n * (r + 1) // world + 1] for r in range(world)]


def consume_checked(capi, shards, truth, bases, offs, device=False):
    """the reads of offs, split among the ranks, into the shards and into the oracle"""
    counted, absorbed = consume(capi, shards, [(bases, o) for o in split(offs, len(shards))], device)
    want = truth.consume_batch(bases, offs, True, nthreads=4)[0]
    assert (counted, absorbed) == (want, want)


def fill(capi, shards, truth, seed, keys_per_shard, round_windows):
    """reads of a genome of their own, in one-round host batches, until each shard holds about
    keys_per_shard keys; returns them"""
    world = len(shards)
    n = -(-int(keys_per_shard * world) // WPR)
    bases = synth_reads(n, L, FAR, seed)
    offs = uniform_offsets(n, L)
    step = world * ((min(round_windows, BATCH_WINDOWS // world) + K - 1) // L)  # window starts per rank <= a round
    for a in range(0, n, step):
        consume_checked(capi, shards, truth, bases, offs[a:min(n, a + step) + 1])
    return bases, offs


def capacities(shards):
    return [s.engine.table.capacity for s in shards]


def assert_filled(shards, cap):
    assert capacities(shards) == [cap] * len(shards)
    for s in shards:
        assert 0.72 * cap <= len(s.engine.table) <= 0.79 * cap, (len(s.engine.table), cap)


def check_exact(shards, truth):
    world = len(shards)
    ks, vs = zip(*[s.local_items_sorted() for s in shards])
    for r, keys in enumerate(ks):
        assert np.all(owner_of(keys, world) == r), "a key sits on a shard that does not own it"
    allk, allv = np.concatenate(ks), np.concatenate(vs)
    order = np.argsort(allk, kind="stable")
    tk, tv = truth.items_sorted()
    assert np.array_equal(allk[order], tk) and np.array_equal(allv[order], tv)
    out = [None] * world

    def red_fn(r):
        def go():
            out[r] = (shards[r].stats(), shards[r].histo(zero=False), shards[r].digest())
        return go

    run_ranks([red_fn(r) for r in range(world)])
    with np.errstate(over="ignore"):
        want_digest = {"n": len(tk), "sum": int(tv.sum(dtype=np.uint64)), "xor": int(np.bitwise_xor.reduce(tk)),
                       "sum_hc": int((tk * tv).sum(dtype=np.uint64)), "foreign": 0}
    want_stats = {"len": len(truth), "sum": truth.sum_counts, "min": truth.min, "max": truth.max}
    want_histo = truth.histo(zero=False)
    for st, hi, dg in out:
        assert st == want_stats
        assert hi == want_histo
        assert dg == want_digest


# ---- 1. a tandem-repeat flood on rank 0 ------------------------------------------------------

HINT_1MI = 300_000       # a shard of 1 Mi slots
HINT_4MI = 1_000_000     # 4 Mi slots: room for the fill and the flood
ROUND_READS = 6990       # reads of 150 bases per rank and round of 1 Mi window starts


def tandem_flood(capi, world, rounds, device, control):
    cap = (4 if control else 1) << 20
    shards = make_shards(capi, world, HINT_4MI if control else HINT_1MI, 1 << 20)
    try:
        assert capacities(shards) == [cap] * world
        truth = OracleTable(K)
        fill(capi, shards, truth, 300 + world, FILL * (1 << 20), 1 << 20)
        if not control:
            assert_filled(shards, cap)
        unit, h = repeat_unit(world, truth.items_sorted()[0])
        assert np.all(owner_of(h, world) == 0)
        # `rounds` rounds of 1 Mi window starts on every rank (a round is counted in window starts,
        # those that straddle two reads included: 6990 reads of 150 bases are 1 Mi less 96), all of
        # their k-mers rank 0's
        bases, offs = repeat_reads(unit, ROUND_READS * rounds)
        assert rounds == -(-(len(bases) - K + 1) // (1 << 20))
        counted, absorbed = consume(capi, shards, [(bases, offs)] * world, device)
        want = sum(truth.consume_batch(bases, offs, True, nthreads=4)[0] for _ in range(world))
        assert (counted, absorbed) == (want, want)
        check_exact(shards, truth)
        after = capacities(shards)
        if control:
            assert after == [cap] * world
        elif world == 4 and rounds == 1:
            # 4 x 1 Mi window starts fit rank 0's deferral list of 4 Mi pairs: the round runs as
            # queued, and the repeat's few new keys need no growth
            assert after == [cap] * world
        else:
            assert after[0] > cap, "the flood never reached growth"
    finally:
        for s in shards:
            s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("rounds", [1, 3])
@pytest.mark.parametrize("world", [4, 8])
def test_tandem_flood_on_one_owner(capi, world, rounds, device):
    tandem_flood(capi, world, rounds, device, control=False)


@pytest.mark.gpu
@pytest.mark.parametrize("rounds", [1, 3])
@pytest.mark.parametrize("world", [4, 8])
def test_tandem_flood_control(capi, world, rounds):
    tandem_flood(capi, world, rounds, False, control=True)


# ---- 2. distinct keys concentrated on one owner -----------------------------------------------

def concentrated(capi, control):
    """world 2, host rounds of 2 Mi window starts: greedy reads of which rank 0 owns about 15/16 of
    the k-mers, two rounds per rank, so the two rounds queued before any is seen bring rank 0 about
    7.5 Mi new keys, more than the room left and its 4 Mi-pair deferral list"""
    world, W = 2, 2 << 20
    cap = (64 if control else 2) << 20
    shards = make_shards(capi, world, 40_000_000 if control else 600_000, W)
    hasher = capi.Table(K)
    try:
        assert capacities(shards) == [cap] * world
        truth = OracleTable(K)
        fill(capi, shards, truth, 500, FILL * (2 << 20), W)
        if not control:
            assert_filled(shards, cap)
        per_round = (W + K - 1) // L  # reads of one rank in a round of W window starts
        n = world * 2 * per_round
        bases, offs = greedy_reads(n, world, 501, hasher.hash_windows)
        share = np.mean(owner_of(read_hashes(bases, n), world) == 0)
        assert share >= 0.9, share
        consume_checked(capi, shards, truth, bases, offs)
        check_exact(shards, truth)
        if control:
            assert capacities(shards) == [cap] * world
        else:
            assert capacities(shards)[0] > cap
    finally:
        hasher.close()
        for s in shards:
            s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("control", [False, True], ids=["burst", "control"])
def test_distinct_keys_concentrated_on_one_owner(capi, control):
    concentrated(capi, control)


# ---- 4. a change of phase ------------------------------------------------------------------------

def phase_change(capi, control):
    """world 2, one host batch of many rounds of 1 Mi window starts per rank: six rounds that only
    repeat keys of the table (the monitor sees nothing made), then ten rounds of new keys.  Once
    the monitor has grown the table, several rounds are queued ahead at a time."""
    world, W = 2, 1 << 20
    cap = (64 if control else 8) << 20
    shards = make_shards(capi, world, 40_000_000 if control else 5_000_000, W)
    try:
        assert capacities(shards) == [cap] * world
        truth = OracleTable(K)
        old, _ = fill(capi, shards, truth, 600, FILL * (8 << 20), W)
        if not control:
            assert_filled(shards, cap)
        per_round = (W + K - 1) // L
        new = synth_reads(world * 10 * per_round, L, FAR, 601)
        parts = []
        for r in range(world):
            rep = old[r * 6 * per_round * L:(r + 1) * 6 * per_round * L]
            fresh = new[r * 10 * per_round * L:(r + 1) * 10 * per_round * L]
            b = np.concatenate([rep, fresh])
            parts.append((b, uniform_offsets(len(b) // L, L)))
        counted, absorbed = consume(capi, shards, parts)
        want = sum(truth.consume_batch(b, o, True, nthreads=4)[0] for b, o in parts)
        assert (counted, absorbed) == (want, want)
        check_exact(shards, truth)
        if control:
            assert capacities(shards) == [cap] * world
        else:
            assert min(capacities(shards)) > cap
    finally:
        for s in shards:
            s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("control", [False, True], ids=["burst", "control"])
def test_change_of_phase_in_one_host_batch(capi, control):
    phase_change(capi, control)


# ---- 3. rounds larger than the small round ---------------------------------------------------

def large_rounds(capi, control):
    """world 2, 8 Mi-window rounds of a device batch (small rounds and deferral lists of 1 Mi and
    4 Mi under OXLI_B200_LAUNCH_MW=1): a round brings each shard about 8 Mi new keys"""
    world, cap = 2, (64 if control else 2) << 20
    shards = make_shards(capi, world, 40_000_000 if control else 600_000, 8 << 20)
    try:
        assert capacities(shards) == [cap] * world
        assert shards[0].engine.info()["round_windows"] == 8 << 20
        truth = OracleTable(K)
        n = -(-int(FILL * (2 << 20) * world) // WPR)
        consume_checked(capi, shards, truth, synth_reads(n, L, FAR, 31), uniform_offsets(n, L), device=True)
        if not control:
            assert_filled(shards, 2 << 20)
        n = world * ((12 << 20) // WPR)  # 12 Mi windows per rank: two rounds
        consume_checked(capi, shards, truth, synth_reads(n, L, FAR, 32), uniform_offsets(n, L), device=True)
        check_exact(shards, truth)
        if control:
            assert capacities(shards) == [cap] * world
        else:
            assert min(capacities(shards)) > cap
    finally:
        for s in shards:
            s.close()


def _large_round_worker(out_path):
    """Runs in a spawned process whose OXLI_B200_LAUNCH_MW is 1: the library reads it once, when it
    loads.  Writes {case: error or null} to out_path."""
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import traceback

    from oxli_b200 import _capi as capi

    results = {}
    for name, control in (("burst", False), ("control", True)):
        try:
            large_rounds(capi, control)
            results[name] = None
        except BaseException:  # noqa: BLE001
            results[name] = traceback.format_exc()
    with open(out_path, "w") as f:
        json.dump(results, f)


@pytest.fixture(scope="module")
def large_round_results(capi, tmp_path_factory):
    import multiprocessing as mp

    out = str(tmp_path_factory.mktemp("large_rounds") / "results.json")
    old = os.environ.get("OXLI_B200_LAUNCH_MW")
    os.environ["OXLI_B200_LAUNCH_MW"] = "1"
    try:
        p = mp.get_context("spawn").Process(target=_large_round_worker, args=(out,))
        p.start()
    finally:
        if old is None:
            del os.environ["OXLI_B200_LAUNCH_MW"]
        else:
            os.environ["OXLI_B200_LAUNCH_MW"] = old
    p.join(timeout=900)
    if p.is_alive():
        p.kill()
        p.join()
    assert p.exitcode == 0, f"the large-round process exited with {p.exitcode}"
    with open(out) as f:
        return json.load(f)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["burst", "control"])
def test_rounds_larger_than_the_small_round(large_round_results, case):
    assert large_round_results[case] is None, large_round_results[case]


@pytest.mark.gpu
def test_bench_shaped_round_into_a_nearly_full_shard(capi):
    """Default constants, 256 Mi-window rounds (bench.py's): one round of 140 Mi windows per rank
    brings each shard more new keys than its 128 Mi-pair deferral list holds.  Too large for the
    CPU oracle: the whole table is checked against one plain table fed the same reads."""
    world, cap, dev = 2, 16 << 20, 0
    shards = make_shards(capi, world, 10_000_000, 256 << 20)
    plain = capi.Table(K, device=dev)
    bufs = []
    try:
        assert capacities(shards) == [cap] * world
        for seed, reads in ((41, -(-int(FILL * cap) // WPR)), (42, (140 << 20) // WPR)):
            # every rank's reads are made on the device, before the ranks start
            parts = []
            for r, s in enumerate(shards):
                d_b = capi.device_alloc(reads * L + 64, s.engine.device)
                d_o = capi.device_alloc((reads + 1) * 8, s.engine.device)
                bufs.append((d_b, d_o, s.engine.device))
                capi.synth_reads_device(d_b, reads, L, FAR, seed, first_read=r * reads, device=s.engine.device)
                capi.h2d(d_o, uniform_offsets(reads, L), s.engine.device)
                parts.append((d_b, d_o))
            if seed == 42:
                assert_filled(shards, cap)
            got = [0] * world

            def rank_fn(r):
                def go():
                    got[r] = shards[r].consume_batch_device(parts[r][0], parts[r][1], reads, reads * L)
                return go

            run_ranks([rank_fn(r) for r in range(world)])
            # the plain table reads the same reads, made again on its own device
            d_b, d_o = capi.device_alloc(reads * L + 64, dev), capi.device_alloc((reads + 1) * 8, dev)
            bufs.append((d_b, d_o, dev))
            capi.h2d(d_o, uniform_offsets(reads, L), dev)
            want = 0
            for r in range(world):
                capi.synth_reads_device(d_b, reads, L, FAR, seed, first_read=r * reads, device=dev)
                st, n, _, _ = plain.consume_batch_device(d_b, d_o, reads, reads * L)
                assert st == 0
                want += n
            assert (sum(got), sum(s.last_absorbed for s in shards)) == (want, want)
        assert min(capacities(shards)) > cap
        out = [None] * world

        def red_fn(r):
            def go():
                out[r] = (shards[r].stats(), shards[r].histo(zero=False), shards[r].digest())
            return go

        run_ranks([red_fn(r) for r in range(world)])
        want_digest = {**plain.device_digest(), "foreign": 0}
        for st, hi, dg in out:
            assert st == plain.stats()
            assert hi == plain.histo()
            assert dg == want_digest
    finally:
        for d_b, d_o, d in bufs:
            capi.device_free(d_b, d)
            capi.device_free(d_o, d)
        plain.close()
        for s in shards:
            s.close()
