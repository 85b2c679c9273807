"""ShardedTable removal (drop / drop_hash / drop_hash_array, mincut / maxcut; src/lib.rs:197-267)
without a GPU: which engine call each method reaches, and the errors raised before any engine call
(a refusal on one rank must not start an exchange the other ranks would wait in)."""
import numpy as np
import pytest

from oxli_b200.sharded import ShardedTable


class FakeTable:
    def __init__(self, ksize):
        self.ksize = ksize

    def hash_windows(self, seq: bytes):
        return np.array([0 if set(seq) - set(b"ACGT") else 1000 + len(seq)], dtype=np.uint64)


class RecordingEngine:
    """the surface of _capi.Shard that removal uses; records each call"""

    def __init__(self, ksize):
        self.table = FakeTable(ksize)
        self.calls = []

    def erase_hashes(self, hashes):
        self.calls.append(("erase_hashes", [int(h) for h in hashes]))
        return 5

    def cut(self, mode, thresh):
        self.calls.append(("cut", mode, thresh))
        return 9


def make(ksize=21):
    return ShardedTable(ksize, 0, 1, engine=RecordingEngine(ksize))


def test_drop_hash_array_sends_the_list():
    t = make()
    assert t.drop_hash_array([3, 2**64 - 1, 3]) == 5
    assert t.engine.calls == [("erase_hashes", [3, 2**64 - 1, 3])]


def test_drop_hash_and_drop_send_one_element_lists_and_return_none():
    t = make(4)
    assert t.drop_hash(77) is None
    assert t.drop("ACGT") is None
    assert t.engine.calls == [("erase_hashes", [77]), ("erase_hashes", [1004])]


def test_cuts_map_to_modes():
    t = make()
    assert t.mincut(2) == 9
    assert t.maxcut(7) == 9
    assert t.engine.calls == [("cut", 0, 2), ("cut", 1, 7)]


def test_drop_of_a_wrong_length_kmer_is_refused_before_any_engine_call():
    t = make(21)
    with pytest.raises(ValueError, match="^kmer size does not match count table ksize$"):
        t.drop("ACGT")
    assert t.engine.calls == []


def test_drop_and_get_refuse_a_non_acgt_kmer_alike():
    t = make(4)
    for call in (t.drop, t.get):
        with pytest.raises(RuntimeError, match="invalid DNA character in input k-mer: ACNT"):
            call("ACNT")
    assert t.engine.calls == []
