"""Pass A of the partitioned pipeline sorts batches of hashes by destination and writes every
destination's run into its fragment (oxli_b200/csrc/scatter.cuh).  These inputs hit the edges of
that design -- a run that crosses the end of its fragment and spills from the middle, groups of
launches that continue fragments at arbitrary fill counts, launches smaller than one batch or
ending inside one, the smallest and largest destination counts, one k per word count of the
specialised kernels -- and compare the table bit for bit with the CPU oracle."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from oracle import OracleTable
from synth import synth_reads, uniform_offsets

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# one k per number of 8-byte words a k-mer takes (2..8), with both sides of the 32/33 split
EVERY_WORD_COUNT = [15, 21, 31, 32, 33, 47, 55, 63]


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


def count_and_compare(capi, k, bases, offs):
    ora = OracleTable(k)
    want, _, _ = ora.consume_batch(bases, offs, True, nthreads=4)
    t = capi.Table(k)
    st, total, er, _ = t.consume_batch(bases, offs, True)
    assert (st, total, er) == (0, want, -1)
    a, b = t.last_consume_pass_ms()
    assert a > 0 and b > 0, "the partitioned pipeline did not run"
    gk, gv = t.export(1)
    ok, ov = ora.items_sorted()
    assert np.array_equal(gk, ok) and np.array_equal(gv, ov), "GPU table differs from the oracle"
    assert t.histo() == ora.histo(zero=False)


def skewed_reads(n_random, n_flood, seed):
    """n_random reads of a random genome, then n_flood reads of a few repeated k-mers (poly-A,
    (AC)n, (ACG)n): their destinations get runs of thousands in every batch, far past frag_cap
    when there are hundreds of destinations"""
    rand = synth_reads(n_random, 150, 300_000, seed=seed)
    motifs = [b"A", b"AC", b"ACG"]
    flood = np.frombuffer(b"".join((motifs[i % 3] * 150)[:150] for i in range(n_flood)), dtype=np.uint8)
    return np.concatenate([rand, flood]), uniform_offsets(n_random + n_flood, 150)


def poly_a_dominated(seed):
    """With two destinations a fragment holds 1.5x its fair share of the launch's windows (plus
    four standard deviations), so only a destination that gets nearly all of them overflows: 5000
    random 150-bp reads and 10 000 poly-A reads of 1000 bp send ~93 % of the windows to poly-A's
    destination, ~1.86x its fair share, and its fragments fill up in the middle of a batch's run."""
    rand = synth_reads(5_000, 150, 300_000, seed=seed)
    bases = np.concatenate([rand, np.frombuffer(b"A" * 1000 * 10_000, dtype=np.uint8)])
    offs = np.concatenate([uniform_offsets(5_000, 150), 5_000 * 150 + np.arange(1, 10_001, dtype=np.uint64) * 1000])
    return bases, offs.astype(np.uint64)


@pytest.mark.parametrize("n_parts", [2, 1024, 2048])
@pytest.mark.parametrize("k", [21, 31, 63])
def test_run_crosses_the_end_of_its_fragment(capi, part, n_parts, k):
    part(n_parts)
    bases, offs = poly_a_dominated(40 + k) if n_parts == 2 else skewed_reads(20_000, 6_000, seed=40 + k)
    count_and_compare(capi, k, bases, offs)


@pytest.mark.parametrize("k", EVERY_WORD_COUNT)
def test_every_word_count(capi, part, k):
    bases = synth_reads(12_000, 150, 200_000, seed=900 + k, sub_ppm=10_000, n_ppm=1_000)
    count_and_compare(capi, k, bases, uniform_offsets(12_000, 150))


# 1 read: one CTA, one tile; 60 and 2000 reads: a grid of a few CTAs or less than one round of the
# full grid; 25 000 reads (3.75 M windows): more than one batch of the full grid, the last one partial
@pytest.mark.parametrize("n_parts", [2, 2048])
@pytest.mark.parametrize("n_reads", [1, 60, 2_000, 25_000])
def test_launch_smaller_than_or_ending_inside_a_batch(capi, part, n_parts, n_reads):
    part(n_parts)
    bases = synth_reads(n_reads, 150, 100_000, seed=n_reads)
    count_and_compare(capi, 31, bases, uniform_offsets(n_reads, 150))


GROUP_SCRIPT = textwrap.dedent("""
    import sys
    sys.path[:0] = [@ROOT@, @TESTS@]
    import numpy as np
    from oracle import OracleTable
    from synth import synth_reads, uniform_offsets
    from oxli_b200 import _capi as capi

    capi.set_pipeline("part", @N_PARTS@, 0)
    n = 36_000  # 5.4 M windows: five or six launches of 1 Mi windows in one group
    bases = synth_reads(n, 150, 400_000, seed=77, sub_ppm=5_000)
    flood = np.frombuffer(b"A" * 150 * 500, dtype=np.uint8)  # one destination spills in every launch
    bases = np.concatenate([bases[: 150 * n // 2], flood, bases[150 * n // 2:]])
    offs = uniform_offsets(n + 500, 150)
    for k in (21, 31, 63):
        ora = OracleTable(k)
        want, _, _ = ora.consume_batch(bases, offs, True, nthreads=4)
        t = capi.Table(k)
        st, total, er, _ = t.consume_batch(bases, offs, True)
        assert (st, total, er) == (0, want, -1), (k, st, total, want, er)
        gk, gv = t.export(1)
        ok, ov = ora.items_sorted()
        assert np.array_equal(gk, ok) and np.array_equal(gv, ov), f"k={k}: GPU table differs from the oracle"
    print("group ok")
""")


@pytest.mark.parametrize("n_parts", [64, 2048])
def test_group_of_launches_continues_fragments(n_parts):
    # Launches of 1 Mi windows (the launch size is read once, when the library loads: a process of
    # its own).  Every launch after the first continues the fragments where the one before left
    # them, at fill counts that are whatever the data made them; each launch also ends inside a
    # batch and is smaller than one batch of the full grid.
    env = dict(os.environ, OXLI_B200_LAUNCH_MW="1", OXLI_B200_ACCUMULATE="8")
    script = (GROUP_SCRIPT.replace("@ROOT@", repr(ROOT)).replace("@TESTS@", repr(os.path.join(ROOT, "tests")))
              .replace("@N_PARTS@", str(n_parts)))
    out = subprocess.run([sys.executable, "-s", "-c", script], env=env, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0 and "group ok" in out.stdout, out.stdout[-2000:] + out.stderr[-4000:]
