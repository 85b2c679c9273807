#!/usr/bin/env python
"""Set operations and cosine of two sharded C3 tables under torchrun (ShardedTable.union /
intersection / difference / symmetric_difference / cosine; oxg_shard_setop_export, oxg_shard_cosine).

The tables: per rank, A counts 12.5 M device-resident reads, as exp_shard.py, and B 12.5 M reads of
which the first half are A's second half (B shares half of A's reads).  Per op: the wall time of the
collective call (it ends synchronised, so the wall time around it is the call's time; the max over
ranks is what the collective call takes), the size of the result, and G slots/s of A plus B scanned.
Also the time of cosine.  Prints the card name and power limit read in the same run.  Rank r runs on
GPU r % (GPUs visible).

PLAIN=lib1:lib2 (at N=1): before the sharded part, oxg_setop_export of two plain tables counted from
the same reads, each library in a process of its own, alternating lib1, lib2, lib1, lib2 (e.g. this
tree's library against the parent commit's, built into an untracked directory).

    PLAIN=oxli_b200/liboxli_b200.so:old/liboxli_b200.so torchrun --standalone --nproc-per-node 1 scripts/exp_shard_setops.py
"""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
n, L, k = int(os.environ.get("READS", 12_500_000)), 150, 21
STEPS = int(os.environ.get("STEPS", 2))
OPS = ("union", "intersection", "difference", "symmetric_difference")
SEED = 0xC30001


def plain_child(lib_path):
    """oxg_setop_export of two plain tables on GPU 0 through the library at lib_path alone (the
    entry points every version of the library has); prints one line"""
    lib = C.CDLL(lib_path)
    vp, u64 = C.c_void_p, C.c_uint64
    for name, args in {"oxg_table_create": [C.c_int, C.c_uint32, u64, C.POINTER(vp)], "oxg_table_destroy": [vp],
                       "oxg_device_alloc": [C.c_int, u64, C.POINTER(vp)], "oxg_device_free": [C.c_int, vp],
                       "oxg_memcpy_h2d": [C.c_int, vp, vp, u64], "oxg_table_len": [vp, C.POINTER(u64)],
                       "oxg_synth_reads_device": [C.c_int, vp, u64, C.c_uint32, u64, u64, u64, C.c_uint32, C.c_uint32],
                       "oxg_consume_batch_device": [vp, vp, vp, u64, u64, C.c_int, C.POINTER(u64), C.POINTER(C.c_int64), C.POINTER(u64)],
                       "oxg_setop_export": [vp, vp, C.c_int, vp, u64, C.POINTER(u64)]}.items():
        getattr(lib, name).argtypes = args
    d_b, d_o = vp(), vp()
    assert lib.oxg_device_alloc(0, n * L + 64, C.byref(d_b)) == 0 and lib.oxg_device_alloc(0, (n + 1) * 8, C.byref(d_o)) == 0
    offs = np.arange(n + 1, dtype=np.uint64) * np.uint64(L)
    assert lib.oxg_memcpy_h2d(0, d_o, offs.ctypes.data, offs.nbytes) == 0
    tabs = []
    for first in (0, n // 2):
        t = vp()
        assert lib.oxg_table_create(0, k, 0, C.byref(t)) == 0
        assert lib.oxg_synth_reads_device(0, d_b, n, L, n, SEED, first, 10_000, 1_000) == 0
        tot, er, ep = u64(), C.c_int64(), u64()
        assert lib.oxg_consume_batch_device(t, d_b, d_o, n, n * L, 1, C.byref(tot), C.byref(er), C.byref(ep)) == 0
        tabs.append(t)
    lens = []
    for t in tabs:
        m = u64()
        assert lib.oxg_table_len(t, C.byref(m)) == 0
        lens.append(m.value)
    out = np.zeros(sum(lens) + 2, dtype=np.uint64)
    res = []
    for op in range(4):
        got = u64()
        ms = []
        for _ in range(STEPS + 1):  # the first call warms up
            t0 = time.perf_counter()
            assert lib.oxg_setop_export(tabs[0], tabs[1], op, out.ctypes.data, len(out), C.byref(got)) == 0
            ms.append(1e3 * (time.perf_counter() - t0))
        res.append(f"{OPS[op]} {min(ms[1:]):.0f} ms ({got.value / 1e6:.1f} M keys)")
    print(f"  plain oxg_setop_export, {lib_path}: |A| {lens[0] / 1e6:.1f} M, |B| {lens[1] / 1e6:.1f} M; " + "; ".join(res), flush=True)
    for t in tabs:
        lib.oxg_table_destroy(t)
    lib.oxg_device_free(0, d_b)
    lib.oxg_device_free(0, d_o)


if len(sys.argv) == 3 and sys.argv[1] == "--plain":
    plain_child(sys.argv[2])
    sys.exit(0)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

sys.path.insert(0, ROOT)
from oxli_b200 import _capi as capi  # noqa: E402
from oxli_b200.sharded import ShardedTable  # noqa: E402

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
local = int(os.environ["LOCAL_RANK"]) % torch.cuda.device_count()
torch.cuda.set_device(local)
dist.init_process_group("gloo")
G = n * world


def exchange(blob):
    out = [None] * world
    dist.all_gather_object(out, blob)
    return out


def mx(x):
    t = torch.tensor([x], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def wall(call):
    """wall seconds of a collective call, max over ranks"""
    dist.barrier()
    t0 = time.perf_counter()
    out = call()
    return mx(time.perf_counter() - t0), out


card = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
cards = [None] * world
dist.all_gather_object(cards, f"{rank}: cuda:{local}, {card}")

plain_lines = []
if os.environ.get("PLAIN") and world == 1:
    for lib_path in os.environ["PLAIN"].split(":") * 2:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--plain", os.path.join(ROOT, lib_path)],
                           capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=str(local)))
        plain_lines.append(r.stdout.strip() or f"  {lib_path}: failed: {r.stderr.strip()[-400:]}")

# the C3-shaped reads: 12.5 M per rank, 1 % substitutions, 0.1 % N, genome 12.5 Mbp x N, k=21
d_b = capi.device_alloc(n * L + 64, local); d_o = capi.device_alloc((n + 1) * 8, local)
offs = np.arange(n + 1, dtype=np.uint64) * np.uint64(L)
capi.h2d(d_o, offs, local)
tables = []
for first in (rank * n, rank * n + n // 2):  # B: the second half of A's reads, then as many new ones
    capi.synth_reads_device(d_b, n, L, G, SEED, first_read=first, sub_ppm=10_000, n_ppm=1_000, device=local)
    t = ShardedTable(k, rank, world, device=local, exchange=exchange)
    t.consume_batch_device(d_b, d_o, n, n * L, True)
    tables.append(t)
A, B = tables
slots = mx(float(A.engine.table.capacity + B.engine.table.capacity))  # (the most any rank scans)
sizes = (A.stats()["len"], B.stats()["len"])
inter, uni = A.setop_sizes(B)

rows = []
for op, name in enumerate(OPS):
    ms = []
    for _ in range(STEPS + 1):  # the first call warms up
        s, (keys, start, total) = wall(lambda: getattr(A, name)(B))
        ms.append(1e3 * s)
    rows.append((name, ms[1:], total))
    del keys
ms_cos = [1e3 * wall(lambda: A.cosine(B))[0] for _ in range(STEPS + 1)][1:]
cos = A.cosine(B)

if rank == 0:
    print(f"cards (rank: device, name, power limit): {cards}", flush=True)
    for line in plain_lines:
        print(line, flush=True)
    print(f"N={world}  C3-shaped tables: |A| {sizes[0] / 1e6:.1f} M, |B| {sizes[1] / 1e6:.1f} M keys, |A&B| {inter / 1e6:.1f} M, "
          f"|A|B| {uni / 1e6:.1f} M; A + B slots on the largest rank {slots / 1e6:.0f} M", flush=True)
    for name, ms, total in rows:
        print(f"  {name}: ms {' '.join(f'{x:.0f}' for x in ms)}; {total / 1e6:.1f} M keys; "
              f"{slots / min(ms) / 1e6:.2f} G slots/s of A + B per rank", flush=True)
    print(f"  cosine: ms {' '.join(f'{x:.1f}' for x in ms_cos)}; value {cos!r}", flush=True)
for t in tables:
    t.close()
for p in (d_b, d_o):
    capi.device_free(p, local)
dist.barrier()
dist.destroy_process_group()
