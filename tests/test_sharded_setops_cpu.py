"""ShardedTable union / intersection / difference / symmetric_difference and cosine (src/lib.rs:610-655,
727-765) without a GPU: which engine call each method reaches, with which op number, that the
engine's answer comes back unchanged, and the TypeError raised before any engine call (a refusal on
one rank must not start an exchange the other ranks would wait in)."""
import numpy as np
import pytest

from oxli_b200.sharded import ShardedTable


class EngineError(RuntimeError):
    """what _capi.check raises: the status of the failed call rides along"""

    def __init__(self, status, msg):
        super().__init__(msg)
        self.status = status


class RecordingEngine:
    """the surface of _capi.Shard that the set operations and cosine use; records each call"""

    def __init__(self, fail=None):
        self.calls = []
        self.fail = fail

    def setop(self, other, op):
        self.calls.append(("setop", other, op))
        if self.fail is not None:
            raise EngineError(self.fail, "refused")
        return np.array([3, 9], dtype=np.uint64), 5, 11

    def cosine(self, other):
        self.calls.append(("cosine", other))
        if self.fail is not None:
            raise EngineError(self.fail, "refused")
        return 0.25


def make(fail=None):
    return ShardedTable(21, 0, 1, engine=RecordingEngine(fail))


def test_each_set_operation_passes_its_op_number():
    a, b = make(), make()
    for name, op in (("union", 0), ("intersection", 1), ("difference", 2), ("symmetric_difference", 3)):
        keys, start, total = getattr(a, name)(b)
        assert keys.tolist() == [3, 9] and start == 5 and total == 11
        assert a.engine.calls[-1] == ("setop", b.engine, op)
    assert len(a.engine.calls) == 4 and b.engine.calls == []


def test_cosine_reaches_the_engine():
    a, b = make(), make()
    assert a.cosine(b) == 0.25
    assert a.engine.calls == [("cosine", b.engine)] and b.engine.calls == []


def test_the_same_table_on_both_sides():
    a = make()
    assert a.intersection(a)[2] == 11
    assert a.engine.calls == [("setop", a.engine, 1)]


def test_other_types_are_refused_before_any_engine_call():
    a = make()
    others = (None, 7, a.engine, object())
    for other in others:
        for call in (a.union, a.intersection, a.difference, a.symmetric_difference, a.cosine):
            with pytest.raises(TypeError, match="ShardedTable"):
                call(other)
    assert a.engine.calls == []


@pytest.mark.parametrize("status, exc", [(2, ValueError), (4, MemoryError), (1, EngineError)])
def test_engine_failures_map_to_python_errors(status, exc):
    a, b = make(fail=status), make()
    for call in (lambda: a.union(b), lambda: a.cosine(b)):
        with pytest.raises(exc, match="refused"):
            call()
