#!/usr/bin/env python
"""bench.py -- canonical k-mers counted per second (BASELINE.json `metric`).

  python bench.py --gpus 1                      C2 = configs[1]: k=31, 10 M x 150-bp reads from a random
                                                5 Mbp genome (~300x coverage), one B200, small hot table
  torchrun ... bench.py --gpus N  (N = 2,4,8)   C3 = configs[2], weak scaling: k=21, 12.5 M reads per GPU
                                                with 1 % substitutions and 0.1 % N from a genome of
                                                12.5 Mbp x N -- at N = 8 exactly the 100 M-read / 100 Mbp
                                                C3; the table is hash-sharded over the N GPUs
  python bench.py --impl reference ...          the CPU restatement of the reference path on this box's
                                                host cores, same config, bounded sample
  python bench.py ... --dump-outputs DIR        also write what the last timed step computed, as .npy
                                                files (one GPU or the reference arm)

A step = build the count table for the whole read set from scratch (clear, consume every read).
One JSON line (rank 0): `value` device-timed with the reads resident in HBM; `e2e` the same job
through the host-buffer C-ABI call (pinned host -> H2D inside the timed region, result read back);
`roofline` the dominant kernels against measured HBM copy bandwidth; `cpu_baseline` the oracle on a
bounded sample (N = 1 only); `parity` the result checked against the oracle after the timed region
(exit code 1 if it does not hold).  torch is the launcher only (process group for the IPC-handle
exchange, barriers and the max over ranks); the product path is the C ABI.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "canonical k-mers counted/sec"
UNIT = "kmers/s"

WORKLOADS = {
    # BASELINE.json configs[1]
    "c2": dict(name="C2", ksize=31, read_len=150, reads=10_000_000, genome=5_000_000, sub_ppm=0, n_ppm=0,
               seed=0xC20001, scale_with_gpus=False),
    # BASELINE.json configs[2], per GPU: at 8 GPUs 100 M reads from a 100 Mbp genome
    "c3": dict(name="C3", ksize=21, read_len=150, reads=12_500_000, genome=12_500_000, sub_ppm=10_000, n_ppm=1_000,
               seed=0xC30001, scale_with_gpus=True),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=[None, "c2", "c3"], help="default: c2 on one GPU, c3 on several")
    ap.add_argument("--reads", type=int, default=0, help="reads per GPU (default: the workload's)")
    ap.add_argument("--genome", type=int, default=0)
    ap.add_argument("--ksize", type=int, default=0)
    ap.add_argument("--cpu-sample-reads", type=int, default=200_000)
    ap.add_argument("--parity-reads", type=int, default=100_000, help="reads per rank of the oracle-checked subsample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--round-mw", type=int, default=256, help="sharded table: Mi windows per round of a device-resident batch "
                    "(the library's default is 64: see DESIGN.md section 6)")
    ap.add_argument("--table-hint", type=int, default=-1, help="expected distinct k-mers (-1: genome length for c2, none for c3)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float64), see dump_outputs()")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def workload(a, world: int) -> dict:
    w = dict(WORKLOADS[a.workload or ("c2" if world == 1 else "c3")])
    if a.reads:
        w["reads"] = a.reads
    if a.genome:
        w["genome"] = a.genome
    if a.ksize:
        w["ksize"] = a.ksize
    w["genome_total"] = w["genome"] * (world if w["scale_with_gpus"] else 1)
    w["reads_total"] = w["reads"] * world
    extras = f", {w['sub_ppm'] / 1e4:g} % substitutions, {w['n_ppm'] / 1e4:g} % N" if w["sub_ppm"] or w["n_ppm"] else ""
    w["label"] = (f"{w['name']}: k={w['ksize']}, {w['reads_total'] / 1e6:g} M x {w['read_len']}-bp reads "
                  f"({w['reads_total'] * w['read_len'] / 1e9:g} Gbp) from a random {w['genome_total'] / 1e6:g} Mbp genome{extras}")
    return w


def measured_peak_gbs() -> tuple[float, str]:
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs.  The poller is
    started early (it needs some hundred ms to produce its first row, more when eight ranks start
    one each) and rows are kept by arrival time: only those that came in between `with` entry and
    exit count."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index
        self.t_in = self.t_out = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
            atexit.register(self.close)  # (a bench that dies before its timed region must not leave the poller behind)
        except Exception:
            self.proc = None

    def __enter__(self):
        self.t_in = time.perf_counter()
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def __exit__(self, *exc):
        self.t_out = time.perf_counter()
        time.sleep(0.12)  # (a row that was being produced when the region ended)
        self.close()

    def close(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
            self.proc = None

    def summary(self) -> dict:
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [r for t, r in self.rows if self.t_in is not None and self.t_in <= t <= (self.t_out or t) + 0.12]
        for r in inside:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for name, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_traffic(name: str):
    """ncu dram__bytes_read+write per k-mer of the dominant kernels (committed capture), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            return json.load(f)[name]
    except Exception:
        return None


DUMP_PAIRS = 1 << 20  # (hash, count) pairs --dump-outputs keeps: 24 MiB of float64


def dump_outputs(out_dir: str, keys: np.ndarray, vals: np.ndarray, histo: list, counted: int) -> None:
    """What a caller of the timed path receives -- the k-mers counted, the (hash, count) table
    sorted by hash, its histogram -- as float64 .npy files, so that two builds can be compared
    output for output.  A table larger than DUMP_PAIRS is sampled at evenly spaced ranks; each
    hash is split into 32-bit halves, which float64 holds exactly."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(keys)
    pick = np.arange(min(n, DUMP_PAIRS), dtype=np.int64) * n // max(min(n, DUMP_PAIRS), 1)
    k, v = keys[pick], vals[pick]
    freq, distinct = np.array(histo, dtype=np.uint64).reshape(-1, 2).T
    arrays = {"kmers_counted": np.array([counted], dtype=np.uint64), "table_size": np.array([n], dtype=np.uint64),
              "table_hash_hi32": k >> np.uint64(32), "table_hash_lo32": k & np.uint64(0xFFFFFFFF), "table_count": v,
              "histo_count": freq, "histo_kmers": distinct}
    for name, x in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), x.astype(np.float64))


def alg_bytes_per_kmer(read_len: int, k: int, world: int = 1) -> float:
    # SURVEY.md 8(d): every base read once (1 B) + 16-B slot read + 8-B count write,
    # + remote 8-B write and read of the routed hash on (N-1)/N of the k-mers
    return read_len / (read_len - k + 1) + 24.0 + 16.0 * (world - 1) / world


# ---------------------------------------------------------------------------------
# reference arm: the oracle port on the box's host cores
# ---------------------------------------------------------------------------------

def run_reference(a, rank: int, world: int):
    """CPU arm: the oracle (C restatement of src/lib.rs:545-607 + sourmash/murmur3) with all host
    threads, on a bounded sample of the same workload.  Rank 0 only."""
    if rank != 0:
        return
    import oracle
    from oracle.synth import synth_reads, uniform_offsets

    w = workload(a, world)
    cores = os.cpu_count() or 1
    # a few seconds of CPU work per step: on C2 (every key seen hundreds of times) the threads' tables stay
    # small and the sample can grow with the cores; on C3 nearly every k-mer is a new key, the port's
    # per-thread tables and their merge (KmerCountTable.add's role) cost 10x more per k-mer
    n = min(w["reads_total"], a.cpu_sample_reads if w["sub_ppm"] else max(a.cpu_sample_reads, 20_000 * cores))
    bases = synth_reads(n, w["read_len"], w["genome_total"], w["seed"], sub_ppm=w["sub_ppm"], n_ppm=w["n_ppm"])
    offs = uniform_offsets(n, w["read_len"])
    times, total = [], 0
    for i in range(a.warmup + a.steps):
        t = oracle.OracleTable(w["ksize"])
        t0 = time.perf_counter()
        total, _, _ = t.consume_batch(bases, offs, True, nthreads=cores)
        dt = time.perf_counter() - t0
        if i >= a.warmup:
            times.append(dt)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, *t.items_sorted(), t.histo(zero=False), total)
    ms = 1e3 * float(np.mean(times))
    v = total / (ms / 1e3)
    sample = f"first {n} reads of the workload ({total} k-mers) per step, table rebuilt each step"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic", "config": config_of(w, world),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "note": "the Rust reference cannot be built here (no cargo/rustc); this is oracle/, "
                                 "its C restatement, reads sharded over threads and merged like KmerCountTable.add"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def config_of(w: dict, world: int) -> dict:
    """The part of `config` both arms share (the driver compares it)."""
    per_gpu = w["reads"] * w["read_len"] / 1e9
    return {"workload": w["label"], "ksize": w["ksize"], "read_len": w["read_len"], "reads": w["reads_total"],
            "genome_len": w["genome_total"], "sub_ppm": w["sub_ppm"], "n_ppm": w["n_ppm"],
            "l2_policy": f"inputs ({per_gpu:.2g} GB of reads per GPU per step) far exceed the 126 MB L2; no flush needed"}


# ---------------------------------------------------------------------------------
# parity
# ---------------------------------------------------------------------------------

def oracle_of(w: dict, first_reads: list[int], n_each: int, skip_bad: bool = True, nthreads: int = 0):
    """Oracle table of reads [f, f + n_each) for every f in first_reads (the generator is a pure
    function of the read index, identical on CPU and GPU: tests/test_gpu_parity.py)."""
    import oracle
    from oracle.synth import synth_reads, uniform_offsets

    t = oracle.OracleTable(w["ksize"])
    total = 0
    for f in first_reads:
        b = synth_reads(n_each, w["read_len"], w["genome_total"], w["seed"], first_read=f, sub_ppm=w["sub_ppm"], n_ppm=w["n_ppm"])
        got = t.consume_batch(b, uniform_offsets(n_each, w["read_len"]), skip_bad, nthreads=nthreads or (os.cpu_count() or 1))
        total += got[0]
        if got[1] >= 0:
            return t, total, (first_reads.index(f), got[1], got[2])
    return t, total, None


def digest_of_pairs(k: np.ndarray, v: np.ndarray) -> dict:
    with np.errstate(over="ignore"):
        return {"n": int(len(k)), "sum": int(v.sum(dtype=np.uint64)), "xor": int(np.bitwise_xor.reduce(k)) if len(k) else 0,
                "sum_hc": int((k * v).sum(dtype=np.uint64))}


def parity_single(a, w, capi, table, d_bases, d_offs, counted: int, dev: int) -> dict:
    """N = 1: (i) the full table's digests through both pipelines, (ii) identities that hold at any
    size, (iii) a subsample table bit for bit against the oracle, skip and error mode."""
    n, L, k = w["reads"], w["read_len"], w["ksize"]
    out = {"ok": True, "checks": []}

    def check(name, ok, **info):
        out["checks"].append({"check": name, "ok": bool(ok), **info})
        out["ok"] = out["ok"] and bool(ok)

    full = table.device_digest()
    hist = table.histo()
    check("sum of counts == k-mers counted", full["sum"] == counted, sum=full["sum"], counted=counted)
    check("sum of histo == distinct, sum f*histo == counted",
          sum(c for _, c in hist) == full["n"] and sum(f * c for f, c in hist) % (1 << 64) == full["sum"])
    capi.set_pipeline("fused")
    other = capi.Table(k, device=dev, capacity_hint=full["n"])
    st, total2, _, _ = other.consume_batch_device(d_bases, d_offs, n, n * L, True)
    capi.set_pipeline("auto")
    d2 = other.device_digest()
    check("fused kernel and partitioned pipeline build the same table (digests, histo)",
          st == 0 and total2 == counted and d2 == full and other.histo() == hist, digest=full)
    other.close()

    m = min(a.parity_reads, n)
    ora, want, _ = oracle_of(w, [0], m)
    sub = capi.Table(k, device=dev)
    st, got, _, _ = sub.consume_batch_device(d_bases, d_offs, m, m * L, True)
    gk, gv = sub.export(1)
    ok_, ov_ = ora.items_sorted()
    check(f"first {m} reads: (hash, count) table bit for bit == oracle", st == 0 and got == want and np.array_equal(gk, ok_)
          and np.array_equal(gv, ov_) and sub.histo() == ora.histo(zero=False), kmers=want, distinct=len(ok_))
    sub.close()
    if w["n_ppm"]:
        ora_e, want_e, err = oracle_of(w, [0], m, skip_bad=False)
        sub = capi.Table(k, device=dev)
        st, got, er, ep = sub.consume_batch_device(d_bases, d_offs, m, m * L, False)
        gk, gv = sub.export(1)
        ok_, ov_ = ora_e.items_sorted()
        check("error mode: counted prefix, read and position == oracle",
              st == capi.ERR_BAD_KMER and err is not None and (er, ep) == (err[1], err[2]) and got == want_e
              and np.array_equal(gk, ok_) and np.array_equal(gv, ov_), read=er, position=ep)
        sub.close()
    return out


# ---------------------------------------------------------------------------------
# one GPU
# ---------------------------------------------------------------------------------

def run_single(a, local: int):
    from oxli_b200 import _capi as capi

    w = workload(a, 1)
    n, L, k = w["reads"], w["read_len"], w["ksize"]
    total_bases = n * L
    dev = local
    d_bases = capi.device_alloc(total_bases + 64, dev)
    d_offs = capi.device_alloc((n + 1) * 8, dev)
    capi.synth_reads_device(d_bases, n, L, w["genome_total"], w["seed"], sub_ppm=w["sub_ppm"], n_ppm=w["n_ppm"], device=dev)
    offs = np.arange(n + 1, dtype=np.uint64) * np.uint64(L)
    capi.h2d(d_offs, offs, dev)
    hint = a.table_hint if a.table_hint >= 0 else (w["genome_total"] if w["name"] == "C2" else 0)
    table = capi.Table(k, device=dev, capacity_hint=hint)
    counted = None

    def step_resident():
        nonlocal counted
        table.clear()
        st, total, _, _ = table.consume_batch_device(d_bases, d_offs, n, total_bases, True)
        assert st == 0 and (counted is None or total == counted), (st, total, counted)
        counted = total
        return table.last_consume_kernel_ms(), table.last_consume_pass_ms()

    clocks = ClockSampler(dev)
    for _ in range(a.warmup):
        step_resident()
    table.sync()
    launches0 = int(capi.lib.oxg_launch_count())
    kernel_ms, kernel_launches, ms_a, ms_b = 0.0, 0, 0.0, 0.0
    with clocks:
        table.timer_start()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            (ms, nl), (pa, pb) = step_resident()
            kernel_ms += ms; kernel_launches += nl; ms_a += pa; ms_b += pb
        dev_ms = table.timer_stop()
        wall_ms = 1e3 * (time.perf_counter() - t0)
    launches = int(capi.lib.oxg_launch_count()) - launches0
    ms_per_step = dev_ms / a.steps
    value = counted / (ms_per_step / 1e3)
    distinct = len(table)
    cap = table.capacity
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, *table.export(1), table.histo(), counted)

    # roofline of the dominant kernels: algorithmic bytes / their own duration, CUDA events on the
    # launch stream.  Partitioned pipeline: scatter_kernel + aggregate_kernel together do what
    # consume_kernel<k,count> does alone, so the pair is the unit.
    peak, peak_src = measured_peak_gbs()
    balg = alg_bytes_per_kmer(L, k)
    partitioned = ms_a > 0
    kernel = (f"scatter_kernel<{k}> + aggregate_kernel (per group of launches)" if partitioned else f"consume_kernel<{k},count>")
    avg_launch_ms = kernel_ms / max(kernel_launches, 1)
    kmers_per_launch = counted * a.steps / max(kernel_launches, 1)
    achieved = balg * kmers_per_launch / (avg_launch_ms / 1e3) / 1e9
    per_kmer = measured_traffic("partitioned_c2" if partitioned else "fused_c2") if w["name"] == "C2" and k == 31 else None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": per_kmer * kmers_per_launch if per_kmer else None,
                "traffic_unit": "bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum, profiles/r2_traffic.json)",
                "alg_bytes_per_launch": balg * kmers_per_launch, "kernel": kernel, "alg_bytes_per_kmer": balg,
                "kmers_per_launch": kmers_per_launch, "avg_launch_ms": avg_launch_ms,
                "kernel_share_of_step": kernel_ms / dev_ms, "peak_source": peak_src,
                "pass_ms_per_step": {"scatter": ms_a / a.steps, "aggregate": ms_b / a.steps} if partitioned else None}

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic",
        "config": config_of(w, 1),
        "details": {"distinct_kmers": distinct, "table_slots": cap, "table_bytes": cap * 16,
                    "pipeline": "partitioned (scatter + aggregate)" if partitioned else "fused (hash + update)",
                    "gbases_per_s": total_bases / (ms_per_step / 1e3) / 1e9},
        "roofline": roofline, "gpu_launches": launches, "wall_ms_per_step": wall_ms / a.steps,
        "clocks": clocks.summary(),
    }

    if not a.no_e2e:
        # same job through the host-buffer entry point: pinned host memory -> H2D inside the timed region
        h_bases = capi.pinned_empty(total_bases)
        capi.d2h(h_bases, d_bases, dev)
        h_offs_raw = capi.pinned_empty((n + 1) * 8)
        h_offs = h_offs_raw.view(np.uint64)
        h_offs[:] = offs

        def step_e2e():
            table.clear()
            st, total, _, _ = table.consume_batch(h_bases, h_offs, True)
            assert st == 0 and total == counted
            return len(table)  # device->host read of the result

        for _ in range(max(1, a.warmup // 2)):
            step_e2e()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            got = step_e2e()
        e2e_ms = 1e3 * (time.perf_counter() - t0) / a.steps
        assert got == distinct
        n_chunks = -(-total_bases // (64 << 20))
        out["e2e"] = {"value": counted / (e2e_ms / 1e3), "unit": UNIT,
                      "h2d_bytes_per_step": int(total_bases + (n + 1) * 8 + n_chunks * 8),
                      "d2h_bytes_per_step": int((n_chunks + 2) * 128),
                      "ms_per_step": e2e_ms, "h2d_gbs": total_bases / (e2e_ms / 1e3) / 1e9,
                      "timing": "host wall clock around the blocking C-ABI call"}
        capi.pinned_free(h_bases); capi.pinned_free(h_offs_raw)

    if not a.no_parity:
        step_resident()
        out["parity"] = parity_single(a, w, capi, table, d_bases, d_offs, counted, dev)
    if not a.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(a, w, capi, d_bases)
    print(json.dumps(out), flush=True)
    if not a.no_parity and not out["parity"]["ok"]:
        sys.exit(1)


def cpu_baseline(a, w, capi, d_bases) -> dict:
    import oracle
    from oracle.synth import uniform_offsets

    n = min(w["reads"], a.cpu_sample_reads)
    bases = np.empty(n * w["read_len"], dtype=np.uint8)
    capi.d2h(bases, d_bases)
    offs = uniform_offsets(n, w["read_len"])
    t = oracle.OracleTable(w["ksize"])
    t0 = time.perf_counter()
    total, _, _ = t.consume_batch(bases, offs, True, nthreads=1)
    dt = time.perf_counter() - t0
    return {"value": total / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"first {n} reads of the same workload ({total} k-mers), single thread like the reference's consume",
            "seconds": dt}


# ---------------------------------------------------------------------------------
# N GPUs: one process per GPU (torchrun), the table hash-sharded over them
# ---------------------------------------------------------------------------------

def run_sharded(a, rank: int, world: int, local: int):
    import torch
    import torch.distributed as dist

    from oxli_b200 import _capi as capi
    from oxli_b200.sharded import BadKmerError, ShardedTable, owner_of

    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))

    def exchange(blob):
        out = [None] * world
        dist.all_gather_object(out, blob)
        return out

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(xs: list[int]) -> list[int]:
        t = torch.tensor(xs, dtype=torch.int64, device=f"cuda:{local}")
        dist.all_reduce(t)
        return [int(v) for v in t.tolist()]

    w = workload(a, world)
    n, L, k = w["reads"], w["read_len"], w["ksize"]
    total_bases = n * L
    first = rank * n
    d_bases = capi.device_alloc(total_bases + 64, local)
    d_offs = capi.device_alloc((n + 1) * 8, local)
    capi.synth_reads_device(d_bases, n, L, w["genome_total"], w["seed"], first_read=first, sub_ppm=w["sub_ppm"],
                            n_ppm=w["n_ppm"], device=local)
    offs = np.arange(n + 1, dtype=np.uint64) * np.uint64(L)
    capi.h2d(d_offs, offs, local)
    hint = a.table_hint if a.table_hint > 0 else 0
    st_table = ShardedTable(k, rank, world, device=local, exchange=exchange, capacity_hint=hint // world if hint else 0,
                            round_windows=a.round_mw << 20)
    shard = st_table.engine
    info = shard.info()
    counted = None

    def step_resident():
        nonlocal counted
        shard.table.clear()
        got = st_table.consume_batch_device(d_bases, d_offs, n, total_bases, True)
        assert counted is None or got == counted
        counted = got
        return shard.last_ms()[0]

    clocks = ClockSampler(local)
    for _ in range(a.warmup):
        step_resident()
    dist.barrier(); torch.cuda.synchronize()
    launches0 = int(capi.lib.oxg_launch_count())
    ev_ms = 0.0
    with clocks:
        t0 = time.perf_counter()
        for _ in range(a.steps):
            ev_ms += step_resident()
        torch.cuda.synchronize(); dist.barrier()
        wall = time.perf_counter() - t0
    launches = int(capi.lib.oxg_launch_count()) - launches0
    ms_per_step = max_over_ranks(ev_ms) / a.steps          # CUDA events on each shard's stream, max over ranks
    wall_ms_per_step = 1e3 * max_over_ranks(wall) / a.steps
    tot_counted, tot_absorbed, tot_launches = sum_over_ranks([counted, st_table.last_absorbed, launches])
    value = tot_counted / (ms_per_step / 1e3)
    stats = st_table.stats()

    e2e = None
    if not a.no_e2e:
        # every rank's reads start in pinned host memory; the call streams them through its staging ring
        h_bases = capi.pinned_empty(total_bases)
        capi.d2h(h_bases, d_bases, local)
        h_offs_raw = capi.pinned_empty((n + 1) * 8)
        h_offs = h_offs_raw.view(np.uint64)
        h_offs[:] = offs

        def step_e2e():
            shard.table.clear()
            got = st_table.consume_batch(h_bases, h_offs, True)
            assert got == counted
            return len(shard.table)  # device -> host read of this shard's result

        step_e2e()
        dist.barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            step_e2e()
        torch.cuda.synchronize(); dist.barrier()
        e2e_ms = 1e3 * max_over_ranks(time.perf_counter() - t0) / a.steps
        rounds = shard.last_ms()[1]
        e2e = {"value": tot_counted / (e2e_ms / 1e3), "unit": UNIT,
               "h2d_bytes_per_step": int(world * (total_bases + (n + 1) * 8 + 8 * rounds)),
               "d2h_bytes_per_step": int(world * (rounds + 4) * 256), "ms_per_step": e2e_ms,
               "h2d_gbs_per_gpu": total_bases / (e2e_ms / 1e3) / 1e9,
               "timing": "barrier + cuda sync both sides, wall clock, max over ranks; oxg_shard_consume_batch from pinned host buffers"}
        capi.pinned_free(h_bases); capi.pinned_free(h_offs_raw)

    parity = None
    if not a.no_parity:
        parity = {"ok": True, "checks": []}

        def check(name, ok, **info_):
            oks = sum_over_ranks([1 if ok else 0])[0] == world
            parity["checks"].append({"check": name, "ok": oks, **info_})
            parity["ok"] = parity["ok"] and oks

        # (i) the full table of the timed workload: digests reduced over the shards inside the library
        step_resident()
        dg = st_table.digest()
        hist = st_table.histo(zero=False)
        check("every key sits on the shard that owns it (full table)", dg["foreign"] == 0)
        check("sum of counts == k-mers counted == k-mers absorbed", dg["sum"] == tot_counted == tot_absorbed,
              sum=dg["sum"], counted=tot_counted, absorbed=tot_absorbed)
        check("sum of histo == distinct, sum f*histo == counted", sum(c for _, c in hist) == dg["n"] == stats["len"]
              and sum(f * c for f, c in hist) % (1 << 64) == dg["sum"], digest=dg)
        # (ii) a subsample of every rank's reads through the same sharded path, against the oracle
        for m, what in ((min(a.parity_reads, n), "digests and histo"), (min(max(a.parity_reads // 10, 1000), n), "bit for bit")):
            sub = ShardedTable(k, rank, world, device=local, exchange=exchange, round_windows=1 << 22)
            got = sub.consume_batch_device(d_bases, d_offs, m, m * L, True)
            ora, want, _ = oracle_of(w, [r * n for r in range(world)], m, nthreads=max(1, (os.cpu_count() or 1) // world))
            want_d = {**ora.digest(), "foreign": 0}
            ok = sum_over_ranks([got])[0] == want and sub.digest() == want_d and sub.histo(zero=False) == ora.histo(zero=False)
            if what == "bit for bit":
                gk, gv = sub.local_items_sorted()
                ok_, ov_ = ora.items_sorted()
                mine = owner_of(ok_, world) == rank
                ok = ok and np.array_equal(gk, ok_[mine]) and np.array_equal(gv, ov_[mine])
            check(f"first {m} reads of every rank: sharded table == oracle ({what})", ok, kmers=want, distinct=want_d["n"])
            if what == "bit for bit" and w["n_ppm"]:
                # error mode, per rank: each rank's reads are counted up to its first bad window
                sub.engine.table.clear()
                try:
                    got = sub.consume_batch_device(d_bases, d_offs, m, m * L, False)
                    mine_err = None
                except BadKmerError as e:
                    got, mine_err = None, (e.read, e.position)
                import oracle as oracle_mod
                from oracle.synth import synth_reads, uniform_offsets
                truth = oracle_mod.OracleTable(k)
                for r in range(world):
                    b = synth_reads(m, L, w["genome_total"], w["seed"], first_read=r * n, sub_ppm=w["sub_ppm"], n_ppm=w["n_ppm"])
                    res = truth.consume_batch(b, uniform_offsets(m, L), False)
                    if r == rank:
                        want_err = (res[1], res[2]) if res[1] >= 0 else None
                gk, gv = sub.local_items_sorted()
                ok_, ov_ = truth.items_sorted()
                mine = owner_of(ok_, world) == rank
                check("error mode per rank: read, position and counted prefixes == oracle (bit for bit)",
                      mine_err == want_err and np.array_equal(gk, ok_[mine]) and np.array_equal(gv, ov_[mine]))
            sub.close()

    # what ONE GPU does with one rank's share of this workload and an unsharded table (the
    # denominator of weak-scaling efficiency; `bench.py --gpus 1` measures C2, another workload)
    single = None
    if rank == 0:
        t1 = capi.Table(k, device=local)
        best = 1e30
        for _ in range(2):
            t1.clear()
            t1.timer_start()
            st, got1, _, _ = t1.consume_batch_device(d_bases, d_offs, n, total_bases, True)
            best = min(best, t1.timer_stop())
        single = {"n_gpus": 1, "value": got1 / (best / 1e3), "unit": UNIT, "ms_per_step": best,
                  "what": f"rank 0's {n} reads alone on one GPU, unsharded table (second of two passes, capacity kept)"}
        t1.close()
    dist.barrier()

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        balg = alg_bytes_per_kmer(L, k, world)
        achieved = balg * value / 1e9
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic",
            "config": config_of(w, world),
            "details": {"reads_per_gpu": n, "distinct_kmers": stats["len"],
                        "sharding": f"hash-high-bits x{world}", "partitions_per_shard": info["n_parts"],
                        "round_windows": info["round_windows"], "exchange_bytes_per_gpu": info["exchange_bytes"],
                        "exchange": "pull: every rank scatters its hashes into fragments per (owner, partition) in its own HBM; "
                                    "the owner's aggregation kernel loads them over NVLink through peer-mapped (CUDA IPC) pointers; "
                                    "rounds are ordered by flags in the exchange headers, awaited on the GPU",
                        "gbases_per_s": world * total_bases / (ms_per_step / 1e3) / 1e9},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak * world, "unit": "GB/s",
                         "frac": achieved / (peak * world), "traffic": None, "alg_bytes_per_kmer": balg,
                         "peak_source": peak_src + f" x {world} GPUs", "scope": "whole step, all ranks",
                         "kernel": f"scatter_kernel<{k}> + aggregate_kernel"},
            "e2e": e2e, "parity": parity, "single_gpu_same_workload": single, "gpu_launches": tot_launches,
            "wall_ms_per_step": wall_ms_per_step,
            "timing": "CUDA events on each shard's stream around its rounds, max over ranks",
            "clocks": clocks.summary(),
        }
        print(json.dumps(out), flush=True)
    st_table.close()
    dist.barrier()
    dist.destroy_process_group()
    if parity is not None and not parity["ok"]:
        sys.exit(1)


def main():
    a = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        return run_reference(a, rank, world)
    if world > 1:
        if a.dump_outputs:
            sys.exit("--dump-outputs: one GPU only (a sharded table's outputs are spread over the ranks)")
        return run_sharded(a, rank, world, local)
    return run_single(a, local)


if __name__ == "__main__":
    main()
