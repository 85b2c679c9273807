"""Pass B of the partitioned pipeline hands out the filled blocks of 128 hashes of a work item's
fragments, laid end to end (oxli_b200/csrc/aggregate.cuh).  These inputs put the edges of that
hand-out in front of it -- fragments whose fill is 0, 1, 127, 128 or 129 (a partition count that
gives ~128 hashes per fragment with either pass A grid: 148 or 296 fragments per partition),
items of a single fragment and items of none (296 items per partition), items whose fragments are
all empty (a hundred reads over 2048 partitions) -- with and without the shared-memory cache,
and compare the table bit for bit with the CPU oracle.  (Fragments filled to frag_cap are in
test_gpu_scatter_batches.py.)"""
import numpy as np
import pytest

from oracle import OracleTable
from synth import synth_reads, uniform_offsets

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def capi():
    from oxli_b200 import _capi

    assert _capi.lib.oxg_device_count() > 0, "GPU tests need a CUDA device"
    return _capi


@pytest.fixture()
def part(capi):
    """force the partitioned pipeline for one test; the knobs go back to automatic afterwards"""
    def choose(n_parts=0, groups=0):
        capi.set_pipeline("part", n_parts, groups)
    choose()
    yield choose
    capi.set_pipeline("auto")


# 20 200 reads of 150 bp = 2.42 M windows of k = 31: 128 per fragment at 128 x 148 or 64 x 296
@pytest.mark.parametrize("n_reads,n_parts,groups", [
    (20_200, 64, 1), (20_200, 128, 1), (20_200, 64, 296), (20_200, 128, 296), (100, 2048, 1), (100, 2048, 5)])
@pytest.mark.parametrize("cache", [True, False])
def test_item_blocks(capi, part, n_reads, n_parts, groups, cache):
    part(n_parts, groups)
    # with the cache: ~30x coverage, so that keys repeat; without: a hint far above the launch
    # tells pass B that nearly every key is new
    bases = synth_reads(n_reads, 150, 5 * n_reads if cache else 3_000_000, seed=n_reads + n_parts + groups)
    offs = uniform_offsets(n_reads, 150)
    ora = OracleTable(31)
    want, _, _ = ora.consume_batch(bases, offs, True, nthreads=4)
    t = capi.Table(31, capacity_hint=0 if cache else 50_000_000)
    st, total, er, _ = t.consume_batch(bases, offs, True)
    assert (st, total, er) == (0, want, -1)
    a, b = t.last_consume_pass_ms()
    assert a > 0 and b > 0, "the partitioned pipeline did not run"
    gk, gv = t.export(1)
    ok, ov = ora.items_sorted()
    assert np.array_equal(gk, ok) and np.array_equal(gv, ov), "GPU table differs from the oracle"
    assert t.histo() == ora.histo(zero=False)
