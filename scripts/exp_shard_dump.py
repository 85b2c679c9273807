#!/usr/bin/env python
"""Export and dump of the sharded C3 table under torchrun (ShardedTable.export / dump;
oxg_shard_export_pairs, oxg_shard_dump).

The table: 12.5 M device-resident reads per rank, as exp_shard.py.  Per sort mode (0 slot order,
1 sortkeys, 2 sortcounts): the wall time of export and of dump (each call ends synchronised, so the
wall time around it is the call's time; the max over ranks is what the collective call takes), the
device time of the length and format kernels (torch.profiler, in a run of its own) as GB/s of text,
and the bytes written.  The file goes to a temporary directory (DUMP_DIR, else the system's) and is
deleted.  At N=1 also the drop-in KmerCountTable.dump (host formatting) of a plain table counted
from the same reads, for comparison.  Prints the card name and power limit read in the same run.
Rank r runs on GPU r % (GPUs visible): with fewer GPUs than ranks, shards share a device, and ranks
that are separate processes on one device time-slice it, so their rate is not a multi-GPU rate.

    torchrun --standalone --nproc-per-node N scripts/exp_shard_dump.py
"""
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oxli_b200 import _capi as capi  # noqa: E402
from oxli_b200.sharded import ShardedTable  # noqa: E402

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
local = int(os.environ["LOCAL_RANK"]) % torch.cuda.device_count()
torch.cuda.set_device(local)
dist.init_process_group("gloo")
n, L, k = int(os.environ.get("READS", 12_500_000)), 150, 21
STEPS = int(os.environ.get("STEPS", 2))
DROPIN = int(os.environ.get("DROPIN", 1 if world == 1 else 0))
G = n * world
FLAGS = {0: {}, 1: {"sortkeys": True}, 2: {"sortcounts": True}}


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

# the C3-shaped reads: 12.5 M per rank, 1 % substitutions, 0.1 % N, genome 12.5 Mbp x N, k=21
d_b = capi.device_alloc(n * L + 64, local); d_o = capi.device_alloc((n + 1) * 8, local)
capi.synth_reads_device(d_b, n, L, G, 0xC30001, first_read=rank * n, sub_ppm=10_000, n_ppm=1_000, device=local)
offs = np.arange(n + 1, dtype=np.uint64) * np.uint64(L)
capi.h2d(d_o, offs, local)
t = ShardedTable(k, rank, world, device=local, exchange=exchange)
t.consume_batch_device(d_b, d_o, n, n * L, True)
size = t.stats()["len"]

tmp = [tempfile.mkdtemp(prefix="oxli_dump_", dir=os.environ.get("DUMP_DIR")) if rank == 0 else None]
dist.broadcast_object_list(tmp, src=0)
tmp = tmp[0]
path = os.path.join(tmp, "counts.tsv")
free_gb = shutil.disk_usage(tmp).free / 1e9

rows = []
for mode, flags in FLAGS.items():
    ms_export = [1e3 * wall(lambda: t.export(**flags))[0] for _ in range(STEPS)]
    ms_dump = []
    for _ in range(STEPS):
        ms_dump.append(1e3 * wall(lambda: t.dump(path, **flags))[0])
    written = os.path.getsize(path) if rank == 0 else 0
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        t.dump(path, **flags)
    kern = {"dump_length_kernel": 0.0, "dump_format_kernel": 0.0}
    for ev in prof.events():
        for name in kern:
            if name in ev.name:
                kern[name] += ev.device_time_total / 1e3  # us -> ms
    kern_ms = [mx(kern["dump_length_kernel"]), mx(kern["dump_format_kernel"])]
    rows.append((mode, ms_export, ms_dump, written, kern_ms))
    dist.barrier()

plain = None
if DROPIN and rank == 0:
    from oxli_b200 import KmerCountTable

    bases = np.zeros(n * L, dtype=np.uint8)
    capi.d2h(bases, d_b, local)
    ref = KmerCountTable(k)
    ref.consume_buffer(bases, offs, True)
    same = len(ref) == size
    t0 = time.perf_counter()
    ref.dump(path, sortkeys=True)
    plain = (1e3 * (time.perf_counter() - t0), os.path.getsize(path), same)
    del ref
dist.barrier()

if rank == 0:
    shutil.rmtree(tmp, ignore_errors=True)
    print(f"cards (rank: device, name, power limit): {cards}", flush=True)
    print(f"N={world}  C3-shaped table: {size / 1e9:.3f} G keys; file in {tmp} ({free_gb:.0f} GB free there), deleted", flush=True)
    for mode, ms_export, ms_dump, written, (ms_len, ms_fmt) in rows:
        print(f"  mode {mode} ({'slot order' if mode == 0 else 'sortkeys' if mode == 1 else 'sortcounts'}): "
              f"export ms {' '.join(f'{x:.0f}' for x in ms_export)}; dump ms {' '.join(f'{x:.0f}' for x in ms_dump)}; "
              f"{written / 1e9:.2f} GB written ({written / min(ms_dump) / 1e6:.2f} GB/s end to end); "
              f"length kernel {ms_len:.1f} ms ({written / world / max(ms_len, 1e-9) / 1e6:.0f} GB/s of text per rank), "
              f"format kernel {ms_fmt:.1f} ms ({written / world / max(ms_fmt, 1e-9) / 1e6:.0f} GB/s per rank)", flush=True)
    if plain:
        print(f"  drop-in KmerCountTable.dump(sortkeys=True) of the same reads on one GPU: {plain[0]:.0f} ms, "
              f"{plain[1] / 1e9:.2f} GB, same length: {plain[2]}", flush=True)
t.close()
for p in (d_b, d_o):
    capi.device_free(p, local)
dist.barrier()
dist.destroy_process_group()
