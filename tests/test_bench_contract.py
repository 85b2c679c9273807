"""bench.py's contract, as far as a box without a GPU can check it: the reference arm's JSON
line (it runs the oracle, the one CPU leg bench.py has), the `config` both arms share, the
workload each GPU count selects, the clock sampler's "rows inside the timed region" rule, and the
arrays --dump-outputs writes (on the GPU as well, for the timed path of one GPU)."""
import json
import os
import subprocess
import sys
import time
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def args(**kw):
    base = dict(gpus=1, steps=1, warmup=0, impl="ours", workload=None, reads=0, genome=0, ksize=0, cpu_sample_reads=2000,
                parity_reads=1000, no_cpu_baseline=True, no_e2e=True, no_parity=True, round_mw=256, table_hint=-1,
                dump_outputs=None)
    base.update(kw)
    return types.SimpleNamespace(**base)


def test_workload_per_gpu_count():
    c2 = bench.workload(args(), 1)
    assert c2["name"] == "C2" and c2["ksize"] == 31 and c2["reads_total"] == 10_000_000 and c2["genome_total"] == 5_000_000
    c3 = bench.workload(args(gpus=8), 8)
    # BASELINE.json configs[2] at eight GPUs: 100 M reads from a 100 Mbp genome, k=21
    assert c3["name"] == "C3" and c3["ksize"] == 21 and c3["reads_total"] == 100_000_000 and c3["genome_total"] == 100_000_000
    assert bench.workload(args(gpus=2), 2)["reads"] == c3["reads"]  # weak scaling: per-GPU work fixed
    cfg = bench.config_of(c3, 8)
    assert cfg["workload"].startswith("C3") and cfg["reads"] == 100_000_000 and "l2_policy" in cfg


def test_algorithmic_bytes():
    # SURVEY.md 8(d): L/(L-k+1) bytes of sequence + 16-B slot read + 8-B count write per k-mer
    assert abs(bench.alg_bytes_per_kmer(150, 31) - (150 / 120 + 24)) < 1e-12
    assert bench.alg_bytes_per_kmer(150, 21, 8) > bench.alg_bytes_per_kmer(150, 21, 1)  # + the routed hash


def oracle_table_of(w: dict, n: int):
    from oracle import OracleTable
    from oracle.synth import synth_reads, uniform_offsets

    t = OracleTable(w["ksize"])
    bases = synth_reads(n, w["read_len"], w["genome_total"], w["seed"], sub_ppm=w["sub_ppm"], n_ppm=w["n_ppm"])
    total, _, _ = t.consume_batch(bases, uniform_offsets(n, w["read_len"]), True, nthreads=4)
    return t, total


def load_dump(d) -> dict:
    names = ("kmers_counted", "table_size", "table_hash_hi32", "table_hash_lo32", "table_count", "histo_count", "histo_kmers")
    out = {name: np.load(os.path.join(d, name + ".npy")) for name in names}
    assert all(x.dtype == np.float64 for x in out.values())
    assert sum(x.nbytes for x in out.values()) <= 64 << 20
    return out


def assert_dump_is_table(d, table, counted: int):
    got = load_dump(d)
    k, v = table.items_sorted()
    assert len(k) <= bench.DUMP_PAIRS and got["table_size"].tolist() == [len(k)]  # kept whole
    keys = (got["table_hash_hi32"].astype(np.uint64) << np.uint64(32)) | got["table_hash_lo32"].astype(np.uint64)
    assert np.array_equal(keys, k) and np.array_equal(got["table_count"].astype(np.uint64), v)
    assert list(zip(got["histo_count"].astype(int).tolist(), got["histo_kmers"].astype(int).tolist())) == table.histo(zero=False)
    assert got["kmers_counted"].tolist() == [counted]


def test_dump_outputs_samples_large_tables_and_keeps_hashes_exact(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_PAIRS", 100)
    keys = np.sort(np.random.default_rng(3).integers(0, 2**64 - 1, size=1000, dtype=np.uint64, endpoint=True))
    keys[-1] = 2**64 - 1
    vals = np.arange(1, 1001, dtype=np.uint64)
    bench.dump_outputs(str(tmp_path), keys, vals, [(1, 999), (2**40, 1)], 12345)
    got = load_dump(tmp_path)
    pick = np.arange(100) * 10
    hi, lo = got["table_hash_hi32"].astype(np.uint64), got["table_hash_lo32"].astype(np.uint64)
    assert np.array_equal((hi << np.uint64(32)) | lo, keys[pick]) and np.array_equal(got["table_count"], vals[pick])
    assert got["table_size"].tolist() == [1000] and got["kmers_counted"].tolist() == [12345]
    assert got["histo_count"].tolist() == [1, 2**40] and got["histo_kmers"].tolist() == [999, 1]


def test_steps_below_one_and_sharded_dumps_are_refused(tmp_path):
    base = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "2"]
    assert subprocess.run(base + ["--steps", "0"], capture_output=True, cwd=ROOT).returncode == 2
    out = subprocess.run(base + ["--dump-outputs", str(tmp_path)], capture_output=True, text=True, cwd=ROOT,
                         env={**os.environ, "WORLD_SIZE": "2"})
    assert out.returncode == 1 and "one GPU only" in out.stderr


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_path_equal_the_oracle(tmp_path):
    """--dump-outputs writes the table the last timed step built: on a workload small enough to be
    kept whole it is the oracle's table, and a second run writes the same arrays."""
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--reads", "20000",
           "--genome", "200000", "--no-e2e", "--no-cpu-baseline", "--parity-reads", "2000"]
    for run in ("a", "b"):
        out = subprocess.run(cmd + ["--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])["steps"] == 2
    table, counted = oracle_table_of(bench.workload(args(reads=20000, genome=200000), 1), 20000)
    assert_dump_is_table(tmp_path / "a", table, counted)
    a, b = load_dump(tmp_path / "a"), load_dump(tmp_path / "b")
    assert all(np.array_equal(a[name], b[name]) for name in a)


def test_reference_arm_prints_the_contract_line(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-sample-reads", "2000", "--workload", "c3", "--reads", "4000", "--genome", "100000",
                          "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == bench.UNIT and d["higher_is_better"] is True
    assert d["value"] > 0 and d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    # same `config` as our arm would print for this command line
    a = args(impl="reference", workload="c3", reads=4000, genome=100000)
    assert d["config"] == bench.config_of(bench.workload(a, 1), 1)
    # --dump-outputs: the oracle table of the 2000-read sample the arm timed
    assert_dump_is_table(tmp_path, *oracle_table_of(bench.workload(a, 1), 2000))


def test_reference_arm_other_ranks_do_nothing(capsys):
    bench.run_reference(args(impl="reference"), rank=1, world=2)
    assert capsys.readouterr().out == ""


def test_clock_rows_outside_the_timed_region_do_not_count():
    c = bench.ClockSampler.__new__(bench.ClockSampler)  # no nvidia-smi here: feed the rows by hand
    c.proc, c.rows = None, []
    row = lambda mhz, cap: [str(mhz), "1965", "700", "0x0", "Not Active", "Not Active", "Not Active", cap]
    now = time.perf_counter()
    c.rows.append((now - 5.0, row(1200, "Active")))      # during warm-up
    c.t_in, c.t_out = now - 1.0, now
    c.rows.append((now - 0.5, row(1965, "Not Active")))  # inside
    c.rows.append((now - 0.2, row(1950, "Not Active")))  # inside
    c.rows.append((now + 3.0, row(600, "Active")))       # long after
    s = c.summary()
    assert s["samples"] == 2 and s["sm_mhz"] == 1957.5 and s["sm_max_mhz"] == 1965.0 and s["reasons"] == []
    c.rows.append((now - 0.1, row(1800, "Active")))
    assert c.summary()["reasons"] == ["sw_power_cap"]
