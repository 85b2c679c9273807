"""ShardedTable.add (KmerCountTable::add, src/lib.rs:778-837) without a GPU: which engine call each
kind of argument reaches, and the errors raised before any engine call (a refusal on one rank
must not start an exchange the other ranks would wait in)."""
import pytest

from oxli_b200.sharded import ShardedTable


class FakeTable:
    def __init__(self, ksize):
        self.ksize = ksize


class RecordingEngine:
    """the surface of _capi.Shard that add uses; records each call"""

    def __init__(self, ksize):
        self.table = FakeTable(ksize)
        self.calls = []

    def merge(self, other):
        self.calls.append(("merge", other))
        return (11, 2)

    def merge_table(self, table):
        self.calls.append(("merge_table", table))
        return (7, 3)


def make(ksize=21, world=1):
    return ShardedTable(ksize, 0, world, engine=RecordingEngine(ksize))


def test_a_sharded_table_is_merged_shard_by_shard():
    a, b = make(), make()
    assert a.add(b) == (11, 2)
    assert a.engine.calls == [("merge", b.engine)] and b.engine.calls == []


def test_a_plain_table_or_none_is_routed():
    a = make()
    t = FakeTable(21)
    assert a.add(t) == (7, 3)
    assert a.add(None) == (7, 3)
    assert a.engine.calls == [("merge_table", t), ("merge_table", None)]


@pytest.mark.parametrize("other", [lambda: make(31), lambda: FakeTable(31)])
def test_another_ksize_is_refused_with_the_reference_message(other):
    a = make(21)
    with pytest.raises(ValueError, match="^KmerCountTables must have the same ksize$"):
        a.add(other())
    assert a.engine.calls == []


def test_adding_a_table_to_itself_is_refused():
    a = make()
    for same in (a, a.engine.table):
        with pytest.raises(ValueError, match="itself"):
            a.add(same)
    assert a.engine.calls == []
