"""Every count-table kernel on keys placed in chosen slots.

The table (csrc/table.cuh) probes linearly from an even home slot, home(key) = top log2(cap)
bits of key * PHI with the low bit cleared, and erase shifts the rest of a run back instead of
leaving tombstones.  Random keys at the loads the table keeps sit in their home bucket almost
always: runs that cross the end of the slot array, or that are hundreds of slots long, then
never occur, and the branches that handle them go untested.  Multiplication by the odd PHI is a
bijection mod 2^64, so a key can be made for any home: key_for(slot, cap, low).  Keys whose
key * PHI share the top 40 bits share one home at every capacity up to 2^40, so growth cannot
separate them: cluster(n, top40).

Each scenario checks the table against the CPU oracle (export, len, stats, histo, and lookups
of every present key plus absent keys with the same homes, which must walk the whole run and
stop at its first empty slot), and asserts the layout it was built for: the capacity the keys
were made for, before and after the operation."""
import random
from collections import defaultdict
from decimal import Decimal, localcontext

import numpy as np
import pytest

import oracle
from oracle import OracleTable

gpu = pytest.mark.gpu

PHI = 0x9E3779B97F4A7C15
PHI_INV = pow(PHI, -1, 1 << 64)
M64 = (1 << 64) - 1
TOP = M64  # the empty-slot marker: as a key it lives in the table's side entry, outside the slots
SMALL_BATCH = 1 << 20  # device hash lists longer than this may defer keys (capi.cu: kSmallBatch)
MAX_PROBE = 1024  # slots a launch with a deferral list walks before it defers (table.cuh: kMaxProbe)


# ---- placing keys --------------------------------------------------------------------------

def lg_of(cap: int) -> int:
    assert cap >= 2 and cap & (cap - 1) == 0, cap
    return cap.bit_length() - 1


def home(key: int, cap: int) -> int:
    """first slot of the key's home bucket in a table of `cap` slots"""
    return (((key * PHI) & M64) >> (64 - lg_of(cap))) & ~1


def key_for(slot: int, cap: int, low: int) -> int:
    """a key homed at the even `slot` of a table of `cap` slots; `low` < 2^(64 - log2 cap) picks
    which one"""
    lg = lg_of(cap)
    assert slot % 2 == 0 and 0 <= slot < cap and 0 <= low < 1 << (64 - lg), (slot, cap, low)
    key = (((slot << (64 - lg)) | low) * PHI_INV) & M64
    if key == TOP:
        raise ValueError("2^64-1 is the empty-slot marker; add it to a test on purpose, not as a slot key")
    return key


def cluster(n: int, top40: int, accept=None) -> list[int]:
    """n distinct keys whose key * PHI share the top 40 bits `top40`: one home at every capacity
    from 2 to 2^40 slots.  accept(key), if given, filters them (by owning shard, say)."""
    assert 0 <= top40 < 1 << 40
    out, low = [], 0
    while len(out) < n:
        assert low < 1 << 24
        key = (((top40 << 24) | low) * PHI_INV) & M64
        low += 1
        if key != TOP and (accept is None or accept(key)):
            out.append(key)
    return out


def top40_at(slot: int, cap: int) -> int:
    """the cluster prefix whose keys are homed at `slot` in a table of `cap` slots"""
    return slot << (40 - lg_of(cap))


def keys_at(slot, cap, n, rr, taken, accept=None):
    """n new keys homed at `slot`, random otherwise"""
    out = []
    while len(out) < n:
        try:
            key = key_for(slot, cap, rr.getrandbits(64 - lg_of(cap)))
        except ValueError:
            continue
        if key not in taken and (accept is None or accept(key)):
            taken.add(key)
            out.append(key)
    return out


def random_keys(n, rr, taken, accept=None):
    out = []
    while len(out) < n:
        key = rr.getrandbits(64)
        if key != TOP and key not in taken and (accept is None or accept(key)):
            taken.add(key)
            out.append(key)
    return out


WRAP = ((-4, 5), (-2, 6), (0, 4), (2, 3))  # (home, keys): 11 keys for the 4 slots before the end


def wrap_keys(cap, rr, taken, accept=None):
    """keys homed at cap-4 and cap-2 (eleven for four slots: their run crosses slot cap-1 -> 0)
    and at 0 and 2, which the wrapped keys push further on"""
    return [k for h, n in WRAP for k in keys_at(h % cap, cap, n, rr, taken, accept)]


def wrap_probes(cap, rr, taken, accept=None):
    """absent keys homed at every bucket the wrapped run covers, and a little beyond"""
    return [k for s in [cap - 4, cap - 2] + list(range(0, 40, 2)) for k in keys_at(s, cap, 2, rr, taken, accept)]


def slots_for(keys: int) -> int:
    """slots of a table grown for `keys` distinct keys (capi.cu: slots_for): at most 50 % load,
    and at most 30 % while the slot array is under 128 MiB"""
    def pow2(x):
        c = 1024
        while c < x:
            c <<= 1
        return c
    cap = pow2(keys + keys // 2 + 1)
    while cap * 16 < 128 << 20 and keys * 10 > cap * 3:
        cap <<= 1
    return max(cap, pow2(2 * keys))


def test_placement_helpers():
    """the helpers against the kernel's home(): a wrapping u64 product in numpy"""
    def home_u64(key, cap):
        with np.errstate(over="ignore"):
            p = np.array([key], dtype=np.uint64) * np.uint64(PHI)
        return int((p >> np.uint64(64 - lg_of(cap)))[0]) & ~1

    rr = random.Random(1)
    for lg in (10, 14, 15, 17, 24, 40, 63):
        cap = 1 << lg
        for slot in (0, 2, cap - 4, cap - 2, rr.randrange(0, cap, 2)):
            for low in (0, 1, (1 << (64 - lg)) - 1, rr.getrandbits(64 - lg)):
                try:
                    key = key_for(slot, cap, low)
                except ValueError:
                    continue
                assert home(key, cap) == home_u64(key, cap) == slot
        # the one (slot, low) that would give 2^64-1 is refused
        v = (TOP * PHI) & M64
        slot, low = v >> (64 - lg), v & ((1 << (64 - lg)) - 1)
        if slot % 2 == 0:
            with pytest.raises(ValueError):
                key_for(slot, cap, low)
    assert home(key_for(16382, 1 << 14, 12345), 1 << 14) == 16382
    keys = [key_for((1 << 14) - 2, 1 << 14, low) for low in range(2000)]
    assert len(set(keys)) == 2000 and {home_u64(k, 1 << 14) for k in keys} == {(1 << 14) - 2}
    # a cluster keeps one home at every capacity; the prefix holding 2^64-1 skips it
    for top40 in (0, 12345 << 14, (1 << 40) - 1, ((TOP * PHI) & M64) >> 24):
        c = cluster(1500, top40)
        assert len(set(c)) == 1500 and TOP not in c
        for lg in range(1, 41):
            assert len({home_u64(k, 1 << lg) for k in c}) == 1
    c = cluster(300, top40_at(6000, 1 << 14), accept=lambda k: k >> 63 == 1)
    assert {home(k, 1 << 14) for k in c} == {6000} and all(k >> 63 == 1 for k in c)
    assert {home(k, 1 << 16) for k in c} == {24000}
    rr = random.Random(2)
    taken = set()
    w = wrap_keys(1 << 14, rr, taken)
    assert [home(k, 1 << 14) for k in w] == [16380] * 5 + [16382] * 6 + [0] * 4 + [2] * 3
    p = wrap_probes(1 << 14, rr, taken)
    assert not set(p) & set(w) and len(set(p)) == len(p)
    assert slots_for(0) == 1024 and slots_for(4000) == 1 << 14 and slots_for(1_200_000) == 1 << 22


# ---- checking ------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def capi():
    from oxli_b200 import _capi

    assert _capi.lib.oxg_device_count() > 0, "GPU tests need a CUDA device"
    return _capi


@pytest.fixture()
def pipeline(capi):
    """force a counting pipeline for one test; back to automatic afterwards"""
    yield capi.set_pipeline
    capi.set_pipeline("auto")


def table_with_cap(capi, cap, k=21):
    t = capi.Table(k, capacity_hint=cap * 3 // 10)
    assert t.capacity == cap
    return t


def ora_add(ora, keys, vals):
    """counts[key] += val, creating the key also for val 0"""
    add = oracle.lib().oxo_table_add_hash
    for key, v in zip(np.asarray(keys, dtype=np.uint64).tolist(), np.asarray(vals, dtype=np.uint64).tolist()):
        add(ora._t, key, v)


def ora_count(ora, occ):
    u, c = np.unique(np.asarray(occ, dtype=np.uint64), return_counts=True)
    ora_add(ora, u, c)


def expected(ok, ov, q):
    """the oracle's count of every query (0 when absent), from its sorted items"""
    q = np.asarray(q, dtype=np.uint64)
    if len(ok) == 0:
        return np.zeros(len(q), dtype=np.uint64)
    i = np.minimum(np.searchsorted(ok, q), len(ok) - 1)
    return np.where(ok[i] == q, ov[i], 0).astype(np.uint64)


def check(t, ora, probes=()):
    gk, gv = t.export(1)
    ok, ov = ora.items_sorted()
    assert len(gk) == len(ok), (len(gk), len(ok))
    assert np.array_equal(gk, ok) and np.array_equal(gv, ov)
    assert len(t) == len(ora)
    assert t.stats() == {"len": len(ora), "sum": ora.sum_counts, "min": ora.min, "max": ora.max}
    assert t.histo() == ora.histo(zero=False)
    probes = np.asarray(probes, dtype=np.uint64)
    assert not np.any(expected(ok, ov, probes)), "a probe meant to be absent is present"
    q = np.concatenate([ok, probes])
    assert np.array_equal(t.get_hashes(q), expected(ok, ov, q))


def assert_wraps(t, cap, keys):
    """the keys of `keys` homed at the last two buckets run on into slots 0, 1, ...: all but the
    four that fit before the end come first in the slot-ordered export"""
    assert t.capacity == cap
    order = t.export(0)[0].tolist()
    high = {k for k in keys if home(k, cap) >= cap - 4}
    assert len(high) > 4
    head = order[: len(order) // 2]
    assert sum(k in high for k in head) >= len(high) - 4


def occurrences(keys, rng, most=3):
    occ = np.repeat(np.asarray(keys, dtype=np.uint64), rng.integers(1, most + 1, len(keys)))
    rng.shuffle(occ)
    return occ


PATHS = ["count_hashes", "count_hashes_fetch", "add_pairs", "set_hash", "device_small", "device_large"]


def load(capi, t, ora, keys, rng, path, most=3):
    """the keys into the table through one insert path, and into the oracle"""
    if path == "set_hash":  # one call per key, some keys twice (the second value replaces the first)
        order = list(keys) + list(keys[::7])
        for key in order:
            v = int(rng.integers(0, 1000))
            t.set_hash(key, v)
            ora.set_hash(key, v)
        return
    occ = occurrences(keys, rng, most)
    if path == "count_hashes":
        t.count_hashes(occ)
        ora_count(ora, occ)
    elif path == "count_hashes_fetch":
        got = t.count_hashes(occ, want_counts=True)
        seen = defaultdict(list)
        for key, c in zip(occ.tolist(), got.tolist()):
            seen[key].append(c)
        # the counts after each of a key's increments, in some order: the oracle's serial counts
        for key, cs in seen.items():
            assert sorted(cs) == [ora.count_hash(key) for _ in cs], key
    elif path == "add_pairs":
        vals = rng.integers(0, 50, len(occ), dtype=np.uint64)
        vals[::5] = 0
        t.add_pairs(occ, vals)
        ora_add(ora, occ, vals)
    else:
        if path == "device_large":  # repeats of the same keys: the table needs no more room
            occ = np.resize(occ, SMALL_BATCH + 4099)
            rng.shuffle(occ)
        assert (len(occ) > SMALL_BATCH) == (path == "device_large")
        d = capi.device_alloc(len(occ) * 8)
        try:
            capi.h2d(d, occ)
            assert t.count_hashes_device(d, len(occ)) == len(occ)
        finally:
            capi.device_free(d)
        ora_count(ora, occ)


# ---- 1. runs that wrap the slot array ---------------------------------------------------------

@gpu
@pytest.mark.parametrize("path", PATHS)
def test_runs_that_wrap_the_slot_array(capi, path):
    cap = 1 << 14
    rr, rng = random.Random(10), np.random.default_rng(10)
    taken = set()
    wrap = wrap_keys(cap, rr, taken)
    keys = wrap + random_keys(500, rr, taken) + [TOP]  # 2^64-1, on purpose: the side entry
    probes = wrap_probes(cap, rr, taken)
    t, ora = table_with_cap(capi, cap), OracleTable(21)
    load(capi, t, ora, keys, rng, path)
    assert_wraps(t, cap, wrap)
    check(t, ora, probes)
    load(capi, t, ora, keys[::-1], rng, path)  # the same keys again, now all present
    assert_wraps(t, cap, wrap)
    check(t, ora, probes)


# ---- 2. long runs below the probe limit -------------------------------------------------------

@gpu
@pytest.mark.parametrize("path", PATHS)
def test_long_runs_below_the_probe_limit(capi, path):
    cap, at = 1 << 15, 6000
    rr, rng = random.Random(20), np.random.default_rng(20)
    both = cluster(1000, top40_at(at, cap))
    run, absent = both[:800], both[800:]  # the absent ones must walk past all 800
    taken = set(both)
    bg = random_keys(400, rr, taken)
    probes = absent + [k for s in range(at, at + 1700, 50) for k in keys_at(s, cap, 1, rr, taken)]
    t, ora = table_with_cap(capi, cap), OracleTable(21)
    # a tenth of the run's keys many times, the rest once to three times
    load(capi, t, ora, run[::10], rng, path, most=40)
    load(capi, t, ora, run + bg, rng, path)
    assert t.capacity == cap and {home(k, cap) for k in run} == {at}
    check(t, ora, probes)

    # growth: the rehash keeps the cluster in one run at its new home
    t.reserve(4 * cap * 3 // 10)
    assert t.capacity == 4 * cap and {home(k, 4 * cap) for k in run} == {4 * at}
    check(t, ora, probes)

    # merge into a table of another capacity that holds part of the run already
    dst, dora = table_with_cap(capi, 1 << 14), OracleTable(21)
    mine = run[300:500] + absent[:100] + random_keys(300, rr, taken)
    vals = rng.integers(0, 9, len(mine), dtype=np.uint64)
    dst.add_pairs(mine, vals)
    ora_add(dora, mine, vals)
    assert dst.merge(t) == dora.add(ora)
    assert dst.capacity == 1 << 14
    check(dst, dora, absent[100:])
    check(t, ora, probes)  # the source is left as it was


# ---- 3. erase across the wrap ---------------------------------------------------------------

class SlotModel:
    """the slot array of a table filled one key at a time (set_hash) and emptied one key at a
    time: linear probing from home(key), erase by backward shift"""

    def __init__(self, cap):
        self.cap, self.slots = cap, {}

    def find(self, key):
        i = home(key, self.cap)
        while i in self.slots:
            if self.slots[i][0] == key:
                return i
            i = (i + 1) % self.cap
        return None

    def set(self, key, v):
        i = self.find(key)
        if i is None:
            i = home(key, self.cap)
            while i in self.slots:
                i = (i + 1) % self.cap
        self.slots[i] = (key, v)

    def erase(self, key):
        hole = self.find(key)
        if hole is None:
            return 0
        del self.slots[hole]
        j = hole
        while True:
            j = (j + 1) % self.cap
            if j not in self.slots:
                return 1
            # the entry at j may fill the hole unless its home lies cyclically in (hole, j]
            if (j - home(self.slots[j][0], self.cap)) % self.cap >= (j - hole) % self.cap:
                self.slots[hole] = self.slots.pop(j)
                hole = j

    def order(self):
        return [self.slots[i] for i in sorted(self.slots)]


def check_model(t, m, probes):
    k, v = t.export(0)  # slot order
    assert list(zip(k.tolist(), v.tolist())) == m.order()
    present = [key for key, _ in m.order()]
    q = np.array(present + probes, dtype=np.uint64)
    want = [val for _, val in m.order()] + [0] * len(probes)
    assert t.get_hashes(q).tolist() == want
    assert len(t) == len(m.slots) and t.capacity == m.cap


@gpu
def test_single_key_erase_across_the_wrap(capi):
    cap = 1 << 14
    rr = random.Random(30)
    taken = set()
    wrap = wrap_keys(cap, rr, taken)
    rr.shuffle(wrap)
    keys = wrap + keys_at(cap - 6, cap, 2, rr, taken) + random_keys(60, rr, taken)
    probes = wrap_probes(cap, rr, taken)
    t, m = table_with_cap(capi, cap), SlotModel(cap)
    for i, key in enumerate(keys):
        t.set_hash(key, i + 1)
        m.set(key, i + 1)
    # the layout: one run from cap-6 across slot cap-1 -> 0
    assert all(s in m.slots for s in list(range(cap - 6, cap)) + list(range(0, 12)))
    assert sum(home(m.slots[s][0], cap) >= cap - 4 for s in range(14)) >= 7
    check_model(t, m, probes)

    def erase_one(key):
        assert t.erase_hashes([key]) == m.erase(key)
        check_model(t, m, probes)

    erase_one(m.slots[cap - 1][0])          # the slot just before the wrap
    erase_one(m.slots[2][0])                # the middle of the wrapped run
    first = cap - 6
    while (first - 1) % cap in m.slots:
        first -= 1
    erase_one(m.slots[first % cap][0])      # the run's first key
    erase_one(probes[0])                    # absent: nothing moves
    rest = [key for key, _ in m.order() if key in set(wrap)]
    rr.shuffle(rest)
    for key in rest:                        # every other wrapped key, one call each
        erase_one(key)
    # several keys in one short list (still the one-thread kernel), with 2^64-1 and an absent key
    t.set_hash(TOP, 9)
    left = [key for key, _ in m.order()][:5]
    assert t.erase_hashes(left + [TOP, probes[1], left[0]]) == 6
    for key in left:
        m.erase(key)
    check_model(t, m, probes + [TOP])


def crafted(capi, cap, rr, rng, at, n_run=700, bg=2000):
    """a table of `cap` slots holding a wrapped run, a run of n_run keys homed at `at`, random
    keys and 2^64-1, with counts 1..20"""
    taken = set()
    wrap = wrap_keys(cap, rr, taken)
    both = cluster(n_run + 200, top40_at(at, cap))
    taken |= set(both)
    keys = wrap + both[:n_run] + random_keys(bg, rr, taken) + [TOP]
    probes = wrap_probes(cap, rr, taken) + both[n_run:]
    vals = rng.integers(1, 21, len(keys), dtype=np.uint64)
    t, ora = table_with_cap(capi, cap), OracleTable(21)
    t.add_pairs(keys, vals)
    ora_add(ora, keys, vals)
    assert_wraps(t, cap, wrap)
    check(t, ora, probes)
    return t, ora, keys, probes, taken


@gpu
def test_bulk_erase_on_wrapped_and_long_runs(capi):
    cap = 1 << 14
    rr, rng = random.Random(31), np.random.default_rng(31)
    t, ora, keys, probes, taken = crafted(capi, cap, rr, rng, 9000)
    wrap, run, bg = keys[:18], keys[18:718], keys[718:-1]
    gone = wrap[::2] + run[::3] + bg[:40] + [TOP]
    lst = gone + gone[:50] + probes[:60] + random_keys(20, rr, taken)  # duplicates and absent keys
    rng.shuffle(lst)
    assert len(lst) >= 256
    assert t.erase_hashes(lst) == len(gone)
    for key in gone:
        ora.drop_hash(key)
    assert t.capacity == cap
    check(t, ora, probes + gone)


@gpu
def test_cuts_on_wrapped_and_long_runs(capi):
    cap = 1 << 14
    rr, rng = random.Random(32), np.random.default_rng(32)
    t, ora, keys, probes, _ = crafted(capi, cap, rr, rng, 100)
    assert t.cut(0, 10) == ora.mincut(10)  # counts below 10 go
    assert t.capacity == cap
    check(t, ora, probes)
    assert t.cut(1, 15) == ora.maxcut(15)  # counts above 15 go
    assert t.capacity == cap
    check(t, ora, probes)


# ---- 4. lookup-only kernels on crafted tables -----------------------------------------------------

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


@gpu
@pytest.mark.parametrize("where", ["a_only", "both"])
def test_set_kernels_on_crafted_tables(capi, where):
    ca, cb = 1 << 14, 1 << 15  # different capacities: A's slot order is not B's
    rr, rng = random.Random(40), np.random.default_rng(40)
    taken = set()
    clus = cluster(1000, top40_at(7000, ca))
    taken |= set(clus)
    wa, wb = wrap_keys(ca, rr, taken), wrap_keys(cb, rr, taken)
    shared = random_keys(300, rr, taken)
    ka = wa + clus[:700] + shared + random_keys(300, rr, taken) + [TOP]
    kb = wb + shared[::2] + wa[::3] + random_keys(400, rr, taken)
    if where == "both":
        kb += clus[300:] + [TOP]
    probes_a, probes_b = clus[700:], clus[:300] if where == "both" else clus
    A, B = table_with_cap(capi, ca), table_with_cap(capi, cb)
    oa, ob = OracleTable(21), OracleTable(21)
    for t, o, keys in ((A, oa, ka), (B, ob, kb)):
        vals = rng.integers(0, 1000, len(keys), dtype=np.uint64)
        t.add_pairs(keys, vals)
        ora_add(o, keys, vals)
    assert A.capacity == ca and B.capacity == cb
    assert_wraps(A, ca, wa)
    assert_wraps(B, cb, wb)
    check(A, oa, probes_a)
    check(B, ob, probes_b + wrap_probes(cb, rr, taken))
    for x, y, ox, oy in ((A, B, oa, ob), (B, A, ob, oa)):
        assert x.setop_sizes(y) == ox.setop_sizes(oy)
        assert x.jaccard(y) == ox.jaccard(oy)
        for op, want in enumerate((ox.union(oy), ox.intersection(oy), ox.difference(oy), ox.symmetric_difference(oy))):
            got = x.setop(y, op).tolist()
            assert len(got) == len(set(got)) and set(got) == want, op
        kx, vx = ox.items_sorted()
        ky, vy = oy.items_sorted()
        _, want = exact_cosine(kx, vx, ky, vy)
        assert_cosine(x.cosine(y), want, len(kx), len(ky))
    assert A.merge(B) == oa.add(ob)
    assert A.capacity == ca
    check(A, oa, probes_a if where == "a_only" else clus[:0])
    check(B, ob, probes_b)


# ---- 5. a cluster past the probe limit ------------------------------------------------------------

@gpu
def test_cluster_past_the_probe_limit(capi):
    """A device list longer than SMALL_BATCH is counted with a deferral list: a key more than
    MAX_PROBE slots past its home is deferred and replayed.  1500 keys of one home at every
    capacity always leave some of them that far out.  The replays must end with every key placed
    and without growing the table for them: the capacity stays within one doubling of what the
    keys need.  A library whose replay loop doubles the table whenever a replay defers again grows
    it here until device memory runs out: never run this test against such a build."""
    rng = np.random.default_rng(50)
    clus = np.array(cluster(1500, 0x5A5A5A5A5A), dtype=np.uint64)
    rnd = rng.integers(0, TOP, 1_200_000, dtype=np.uint64)
    occ = np.concatenate([rnd, clus, clus[::3], clus[::7]])
    rng.shuffle(occ)
    assert len(occ) > SMALL_BATCH and len(clus) > MAX_PROBE + 400
    t, ora = capi.Table(21), OracleTable(21)
    d = capi.device_alloc(len(occ) * 8)
    try:
        capi.h2d(d, occ)
        st = capi.lib.oxg_count_hashes_device(t.handle, d, len(occ), 0, None)
    finally:
        capi.device_free(d)
    assert st == capi.OK, capi.lib.oxg_last_error()
    ora_count(ora, occ)
    assert t.capacity <= 2 * slots_for(len(ora)), (t.capacity, len(ora))
    check(t, ora, cluster(1600, 0x5A5A5A5A5A)[1500:])


# ---- 6. consume with k-mers chosen by their hash ---------------------------------------------------

_chosen = {}


def kmers_homed_last(k):
    """a few hundred k-mers of a random sequence whose hash h has h * PHI with the top 14 bits all
    ones: homed at the last bucket (slots cap-2, cap-1) of a 2^15-slot table, and all in one
    bucket of pass B's shared-memory table whatever the partition"""
    if k not in _chosen:
        rng = np.random.default_rng(60 + k)
        seq = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, 6_000_000)]
        h = oracle.hash_windows(seq, k)
        with np.errstate(over="ignore"):
            top = (h * np.uint64(PHI)) >> np.uint64(50)
        at = np.nonzero((top == (1 << 14) - 1) & (h != 0))[0]
        _, first = np.unique(h[at], return_index=True)
        _chosen[k] = [seq[i:i + k].tobytes() for i in np.sort(at[first])]
    return _chosen[k]


def revcomp(s: bytes) -> bytes:
    return s[::-1].translate(bytes.maketrans(b"ACGT", b"TGCA"))


@gpu
@pytest.mark.parametrize("k", [21, 31])
@pytest.mark.parametrize("choice", ["fused", "part"])
def test_consume_kmers_chosen_by_hash(capi, pipeline, k, choice):
    pipeline(choice, 2 if choice == "part" else 0)
    cap = 1 << 15
    kmers = kmers_homed_last(k)
    assert 250 <= len(kmers) <= 600
    rng = np.random.default_rng(61)
    reads = []
    for i, s in enumerate(kmers):  # each k-mer one to five times, forward or reverse complement
        reads += [s if (i + j) % 2 else revcomp(s) for j in range(int(rng.integers(1, 6)))]
    reads += [np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, 150)].tobytes() for _ in range(5)]
    order = rng.permutation(len(reads))
    reads = [reads[i] for i in order]
    # a consume call reserves room for as many keys as its batch has bases: batches of at most
    # 5000 bases keep the table at 2^15 slots
    batches, at = [], 0
    while at < len(reads):
        end, n = at, 0
        while end < len(reads) and n + len(reads[end]) <= 5000:
            n += len(reads[end])
            end += 1
        part = reads[at:end]
        batches.append((np.frombuffer(b"".join(part), dtype=np.uint8),
                        np.concatenate([[0], np.cumsum([len(r) for r in part])]).astype(np.uint64)))
        at = end
    ora = OracleTable(k)
    t = table_with_cap(capi, cap, k)
    # absent keys homed at cap-2 and in the buckets past slot 0: lookups walk the wrapped run
    probes = wrap_probes(cap, random.Random(62 + k), set())
    hashes = oracle.hash_windows(np.frombuffer(b"".join(kmers), dtype=np.uint8), k)[::k].tolist()
    assert {home(h, cap) for h in hashes} == {cap - 2}
    for rep in range(2):  # the second time every key is present already
        for bases, offs in batches:
            want, _, _ = ora.consume_batch(bases, offs, True)
            st, total, er, _ = t.consume_batch(bases, offs, True)
            assert (st, total, er) == (0, want, -1)
            if choice == "part":
                assert t.last_consume_pass_ms()[0] > 0, "the partitioned pipeline did not run"
            assert t.capacity == cap
        assert_wraps(t, cap, hashes)
        check(t, ora, probes)


# ---- 7. shard lookup on crafted tables ------------------------------------------------------------

def run_ranks(fns):
    """one thread per rank; re-raise the first failure"""
    import threading

    errs = [None] * len(fns)

    def wrap(i):
        try:
            fns[i]()
        except BaseException as e:  # noqa: BLE001
            errs[i] = e

    ts = [threading.Thread(target=wrap, args=(i,)) for i in range(len(fns))]
    for th in ts:
        th.start()
    for th in ts:
        th.join(timeout=300)
    assert not any(th.is_alive() for th in ts), "a rank hung"
    for e in errs:
        if e is not None:
            raise e


@gpu
def test_shard_lookup_on_crafted_tables(capi):
    """Two shards on one GPU, each holding keys it owns (top bit = rank) in a wrapped run and a
    700-key run: the collective lookup from both ranks must answer every key, and the absent keys
    homed in those runs with 0.  The shards are fresh: no consume or lookup ran on them before."""
    from oxli_b200.sharded import ShardedTable

    world, cap = 2, 1 << 14
    n_dev = capi.lib.oxg_device_count()
    shards = ShardedTable.local(21, world, [r % n_dev for r in range(world)], capacity_hint=cap * 3 // 10,
                                round_windows=1 << 16)
    rr, rng = random.Random(70), np.random.default_rng(70)
    truth, probes, taken = {}, [], set()
    for r, s in enumerate(shards):
        t = s.engine.table
        assert t.capacity == cap  # the capacity the keys are made for
        own = (lambda r: lambda key: key >> 63 == r)(r)  # the top bit picks the owner of two
        wrap = wrap_keys(cap, rr, taken, own)
        run = cluster(900, top40_at(cap // 2, cap), own)
        taken |= set(run)
        keys = wrap + run[:700] + random_keys(300, rr, taken, own)
        vals = rng.integers(0, 100, len(keys), dtype=np.uint64)
        t.add_pairs(keys, vals)
        truth.update(zip(keys, vals.tolist()))
        probes += wrap_probes(cap, rr, taken, own) + run[700:]
        assert_wraps(t, cap, wrap)
    q = np.array(list(truth) + probes + [0, TOP], dtype=np.uint64)
    rng.shuffle(q)
    queries = [q[: len(q) // 3], q[len(q) // 3:]]  # lists of different sizes, each with keys of both owners
    got = [None] * world

    def go(r):
        got[r] = shards[r].get_hash_array(queries[r])

    run_ranks([lambda r=r: go(r) for r in range(world)])
    for qs, a in zip(queries, got):
        assert a.tolist() == [truth.get(key, 0) for key in qs.tolist()]
    for s in shards:
        assert s.engine.table.capacity == cap
        s.close()


# ---- 8. scan edges ------------------------------------------------------------------------------

@gpu
def test_scans_at_their_edges(capi):
    """histo with more counts of 2^16 and above than its first list holds (the scan runs again
    with a longer one), counts in every bin range up to 2^64-1, a sum that wraps past 2^64 (the
    reference sums in u64), the count sort over all eight byte passes and a short export"""
    rr, rng = random.Random(80), np.random.default_rng(80)
    taken = set()
    # run_stats lists counts >= 2^16 in a buffer of the device context that starts at 2^16 entries
    # and only ever grows: its retry is taken here as long as no earlier test in the process
    # listed more than this many such counts (none does)
    big = random_keys(300_000, rr, taken)
    mid = random_keys(3000, rr, taken)
    small = random_keys(3000, rr, taken)
    edge = random_keys(5, rr, taken)
    keys = big + mid + small + edge + [TOP]
    vals = np.concatenate([
        rng.integers(1 << 16, 1 << 58, len(big), dtype=np.uint64),  # listed raw
        rng.integers(1024, 1 << 16, len(mid), dtype=np.uint64),     # dense global bins
        rng.integers(0, 1024, len(small), dtype=np.uint64),         # shared-memory bins
        np.array([M64, 1 << 63, 1 << 63, 65535, 1024], dtype=np.uint64),
        np.array([70_000], dtype=np.uint64),                       # 2^64-1's own count
    ])
    t, ora = capi.Table(21), OracleTable(21)
    t.add_pairs(keys, vals)
    ora_add(ora, keys, vals)
    assert sum(vals.tolist()) > M64  # the sum wraps
    check(t, ora)
    assert t.stats()["sum"] == sum(vals.tolist()) & M64

    ok, ov = ora.items_sorted()
    by_count = np.lexsort((ok, ov))  # by count, ties by hash
    gk, gv = t.export(2)
    assert np.array_equal(gk, ok[by_count]) and np.array_equal(gv, ov[by_count])

    # a buffer shorter than the table: only the first `cap` pairs are written
    n = len(ok)
    for mode, (wk, wv) in ((1, (ok, ov)), (2, (ok[by_count], ov[by_count]))):
        short = n // 3
        kb = np.full(n, 7, dtype=np.uint64)
        vb = np.full(n, 7, dtype=np.uint64)
        n_out = capi.u64()
        capi.check(capi.lib.oxg_export(t.handle, kb.ctypes.data, vb.ctypes.data, short, mode, capi.C.byref(n_out)))
        assert n_out.value == n
        assert np.array_equal(kb[:short], wk[:short]) and np.array_equal(vb[:short], wv[:short])
        assert not np.any(kb[short:] != 7) and not np.any(vb[short:] != 7)


# ---- 9. cosine against an exact reference -------------------------------------------------------

@gpu
def test_cosine_against_exact_reference(capi):
    """About 10^6 keys a table with counts up to 2^31, against the cosine computed from exact
    integer sums.  The dot product is kept below 2^64: the reference sums it in u64, and how its
    result behaves once that sum wraps is not something a 40-digit reference can stand in for, so
    the wrapped case is left out here."""
    rng = np.random.default_rng(90)
    keys = np.unique(rng.integers(0, TOP, 2_000_000, dtype=np.uint64))
    keys = keys[keys != np.uint64(TOP)]
    rng.shuffle(keys)
    shared, a_only, b_only = keys[:500_000], keys[500_000:1_000_000], keys[1_000_000:1_400_000]
    top = np.uint64((1 << 31) - 1)
    va_s = rng.integers(0, 1 << 20, len(shared), dtype=np.uint64)
    vb_s = rng.integers(0, 1 << 20, len(shared), dtype=np.uint64)
    va_s[:2] = top
    vb_s[:2] = top
    side = np.array([TOP], dtype=np.uint64)  # 2^64-1 in both: the side entries' product joins the dot
    ka = np.concatenate([shared, a_only, side])
    va = np.concatenate([va_s, rng.integers(0, 1 << 31, len(a_only), dtype=np.uint64), np.array([12345], dtype=np.uint64)])
    kb = np.concatenate([shared, b_only, side])
    vb = np.concatenate([vb_s, rng.integers(0, 1 << 31, len(b_only), dtype=np.uint64), np.array([678], dtype=np.uint64)])
    dot, want = exact_cosine(ka, va, kb, vb)
    assert dot < 1 << 64
    A, B = capi.Table(21), capi.Table(21)
    A.add_pairs(ka, va)
    B.add_pairs(kb, vb)
    assert len(A) == len(ka) and len(B) == len(kb)
    assert_cosine(A.cosine(B), want, len(ka), len(kb))
    assert_cosine(B.cosine(A), want, len(kb), len(ka))
