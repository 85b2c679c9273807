#!/usr/bin/env python
"""Adding a plain table into the sharded C3 table under torchrun (ShardedTable.add, oxg_shard_merge_table).

Each rank counts a C3-shaped plain table on its own GPU from READS (12.5 M) device-resident reads of
another seed (another genome: nearly every key is new to the sharded table), and the sharded table
consumes its usual C3 share.  Every call adds into a fresh copy of the sharded table (consumed
again), so each one routes, grows once and adds the same pairs.  A call ends synchronised, so the
wall time around it is the call's time; the max over ranks is what the collective add takes.
Prints G pairs/s per rank and in total, the card name, power limit and max SM clock read in the same
run, and at N=1 also oxg_merge of the same two tables (the shard's own table, no routing).  Rank r
runs on GPU r % (GPUs visible): with fewer GPUs than ranks, shards share a device, and ranks that are
separate processes on one device time-slice it, so their rate is not a multi-GPU rate.

    torchrun --standalone --nproc-per-node N scripts/exp_shard_merge.py
"""
import os
import subprocess
import sys
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
WARMUP, STEPS = 1, int(os.environ.get("STEPS", 3))
G = n * world


def exchange(blob):
    out = [None] * world
    dist.all_gather_object(out, blob)
    return out


def mx(x):
    t = torch.tensor([x], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


card = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
cards = [None] * world
dist.all_gather_object(cards, f"{rank}: cuda:{local}, {card}")

# reads: the C3 share (12.5 M reads per rank, 1 % substitutions, 0.1 % N, genome 12.5 Mbp x N, k=21)
# and the same shape from another seed for the plain table
d_b = capi.device_alloc(n * L + 64, local); d_o = capi.device_alloc((n + 1) * 8, local)
capi.h2d(d_o, np.arange(n + 1, dtype=np.uint64) * np.uint64(L), local)
capi.synth_reads_device(d_b, n, L, G, 0xC30002, first_read=rank * n, sub_ppm=10_000, n_ppm=1_000, device=local)
src = capi.Table(k, local)
src.consume_batch_device(d_b, d_o, n, n * L, True)
pairs = len(src)
capi.synth_reads_device(d_b, n, L, G, 0xC30001, first_read=rank * n, sub_ppm=10_000, n_ppm=1_000, device=local)


def fresh():
    t = ShardedTable(k, rank, world, device=local, exchange=exchange)
    t.consume_batch_device(d_b, d_o, n, n * L, True)
    return t


def timed(call):
    """wall ms of call(t) on a fresh sharded table, max over ranks; warm-up calls first"""
    ms, t = [], None
    for i in range(WARMUP + STEPS):
        if t is not None:
            t.close()
        t = fresh()
        dist.barrier()
        t0 = time.perf_counter()
        call(t)
        wall = mx(time.perf_counter() - t0)
        if i >= WARMUP:
            ms.append(1e3 * wall)
    return ms, t


ms_add, t = timed(lambda t: t.add(src))
d_add = t.digest()
size, cap = t.stats()["len"], t.engine.table.capacity
t.close()
plain = None
if world == 1:
    ms_plain, tp = timed(lambda t: t.engine.table.merge(src))
    plain = (ms_plain, tp.digest() == d_add)
    tp.close()
all_pairs = [None] * world
dist.all_gather_object(all_pairs, (pairs, cap))
if rank == 0:
    total = sum(p[0] for p in all_pairs)
    best = min(ms_add)
    print(f"cards (rank: device, name, power limit, max SM clock): {cards}", flush=True)
    print(f"N={world}  plain tables of {[p[0] for p in all_pairs]} keys added into the C3-shaped sharded table; "
          f"after: {size / 1e9:.3f} G keys, slots per shard {[p[1] for p in all_pairs]}", flush=True)
    print("  ShardedTable.add, ms per call (max over ranks): " + " ".join(f"{x:.1f}" for x in ms_add)
          + f"  -> best {total / world / best / 1e6:.2f} G pairs/s per rank, {total / best / 1e6:.2f} G pairs/s in total", flush=True)
    if plain:
        print("  oxg_merge of the same tables (no routing): " + " ".join(f"{x:.1f}" for x in plain[0])
              + f"  -> best {total / min(plain[0]) / 1e6:.2f} G pairs/s; same table: {plain[1]}", flush=True)
src.close()
for p in (d_b, d_o):
    capi.device_free(p, local)
dist.barrier()
dist.destroy_process_group()
