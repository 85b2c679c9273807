"""ShardedTable export / dump (src/lib.rs:330-381) without a GPU: which engine call each method
reaches, with which sort mode, and the both-flags error raised before any engine call (a refusal on
one rank must not start an exchange the other ranks would wait in)."""
import numpy as np
import pytest

from oxli_b200.sharded import ShardedTable


class RecordingEngine:
    """the surface of _capi.Shard that export and dump use; records each call"""

    def __init__(self):
        self.calls = []

    def export_pairs(self, sort_mode):
        self.calls.append(("export_pairs", sort_mode))
        return np.array([4], dtype=np.uint64), np.array([1], dtype=np.uint64), np.array([[0, 1]], dtype=np.uint64), 1

    def dump(self, path, sort_mode):
        self.calls.append(("dump", path, sort_mode))


def make():
    return ShardedTable(21, 0, 1, engine=RecordingEngine())


def test_export_maps_the_flags_to_sort_modes():
    t = make()
    k, v, runs, total = t.export()
    assert k.tolist() == [4] and v.tolist() == [1] and runs.tolist() == [[0, 1]] and total == 1
    t.export(sortkeys=True)
    t.export(sortcounts=True)
    assert t.engine.calls == [("export_pairs", 0), ("export_pairs", 1), ("export_pairs", 2)]


def test_dump_passes_the_path_and_the_sort_mode():
    t = make()
    assert t.dump("/x/counts.tsv") is None
    t.dump("b.tsv", sortkeys=True)
    t.dump("c.tsv", sortcounts=True)
    assert t.engine.calls == [("dump", "/x/counts.tsv", 0), ("dump", "b.tsv", 1), ("dump", "c.tsv", 2)]


def test_both_flags_are_refused_before_any_engine_call():
    t = make()
    for call in (lambda: t.export(sortcounts=True, sortkeys=True), lambda: t.dump("a.tsv", sortcounts=True, sortkeys=True)):
        with pytest.raises(ValueError, match=r"^Cannot sort by both counts and keys at the same time\.$"):
            call()
    assert t.engine.calls == []
