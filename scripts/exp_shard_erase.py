#!/usr/bin/env python
"""Removing keys from the sharded C3 table under torchrun (ShardedTable.mincut, drop_hash_array,
drop_hash; oxg_shard_cut, oxg_shard_erase_hashes*).

Every call removes keys, so each one runs on a fresh copy of the table (12.5 M device-resident reads
per rank, as exp_shard.py, consumed again).  Timed: mincut(2) (and the share of keys it removes),
drop_hash_array of KEYS (64 Mi) hashes per rank from device lists, half present keys hashed from the
rank's own reads, half uniform random u64 (mark + rebuild path), and one drop_hash per rank (walk
path).  A call ends synchronised, so the wall time around it is the call's time; the max over ranks
is what the collective call takes.  At N=1 also the plain table's oxg_cut / oxg_erase_hashes (host
list) on the same table.  Prints the card name and power limit read in the same run.  Rank r runs on
GPU r % (GPUs visible): with fewer GPUs than ranks, shards share a device, and ranks that are separate
processes on one device time-slice it, so their rate is not a multi-GPU rate.

    torchrun --standalone --nproc-per-node N scripts/exp_shard_erase.py
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
Q = int(os.environ.get("KEYS", 64 << 20))
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


card = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
cards = [None] * world
dist.all_gather_object(cards, f"{rank}: cuda:{local}, {card}")

# the C3-shaped reads: 12.5 M per rank, 1 % substitutions, 0.1 % N, genome 12.5 Mbp x N, k=21
d_b = capi.device_alloc(n * L + 64, local); d_o = capi.device_alloc((n + 1) * 8, local)
capi.synth_reads_device(d_b, n, L, G, 0xC30001, first_read=rank * n, sub_ppm=10_000, n_ppm=1_000, device=local)
capi.h2d(d_o, np.arange(n + 1, dtype=np.uint64) * np.uint64(L), local)


def fresh():
    t = ShardedTable(k, rank, world, device=local, exchange=exchange)
    t.consume_batch_device(d_b, d_o, n, n * L, True)
    return t


def timed(call):
    """wall ms of call(t) on a fresh table, max over ranks; the first WARMUP calls are not kept.
    Returns the times and the last call's result."""
    ms, out = [], None
    for i in range(WARMUP + STEPS):
        t = fresh()
        dist.barrier()
        t0 = time.perf_counter()
        out = call(t)
        wall = mx(time.perf_counter() - t0)
        t.close()
        if i >= WARMUP:
            ms.append(1e3 * wall)
    return ms, out


t = fresh()
size = t.stats()["len"]
slot_bytes = t.engine.table.capacity * 16
# the list: present keys from this rank's reads (windows across a read boundary or an N hash to 0:
# dropped), uniform random u64 for the other half
half = Q // 2
n_hr = min(n, half // (L - k + 1) * 5 // 4 + 1)
d_h = capi.device_alloc(n_hr * L * 8, local)
t.engine.table.hash_batch_device(d_b, d_o, n_hr, n_hr * L, d_h)
h = np.zeros(n_hr * L - k + 1, dtype=np.uint64)
capi.d2h(h, d_h, local)
capi.device_free(d_h, local)
t.close()
present = h[h != 0][:half]
assert len(present) == half
rng = np.random.default_rng(1000 + rank)
q = rng.permutation(np.concatenate([present, rng.integers(0, (1 << 64) - 1, Q - half, dtype=np.uint64, endpoint=True)]))
d_q = capi.device_alloc(Q * 8, local)
capi.h2d(d_q, q, local)

ms_cut, cut_removed = timed(lambda t: t.mincut(2))
ms_list, list_removed = timed(lambda t: t.engine.erase_hashes_device(d_q, Q))
ms_one, _ = timed(lambda t: t.drop_hash(int(present[rank])))
plain = None
if world == 1:
    # context: the shard's own table cut and erased directly (no routing; the list from host memory)
    ms_pcut, pcut = timed(lambda t: t.engine.table.cut(0, 2))
    ms_perase, perase = timed(lambda t: t.engine.table.erase_hashes(q))
    plain = (ms_pcut, pcut == cut_removed, ms_perase, perase == list_removed)
sizes = [None] * world
dist.all_gather_object(sizes, slot_bytes)

if rank == 0:
    total = size  # (stats() is collective: len of the whole table)
    print(f"cards (rank: device, name, power limit): {cards}", flush=True)
    print(f"N={world}  C3-shaped table: {total / 1e9:.3f} G keys, {[round(b / 2**30, 1) for b in sizes]} GiB of slots per shard", flush=True)
    print("ms per call, max over ranks, each on a fresh table:", flush=True)
    print("  mincut(2) " + " ".join(f"{x:.1f}" for x in ms_cut)
          + f"  -> {cut_removed} keys removed ({cut_removed / total:.3f} of the table)", flush=True)
    print(f"  drop_hash_array, {Q} device-resident keys per rank (half present) " + " ".join(f"{x:.1f}" for x in ms_list)
          + f"  -> {list_removed} keys removed; best {world * Q / min(ms_list) / 1e6:.2f} G keys/s in total", flush=True)
    print("  drop_hash, one key per rank " + " ".join(f"{x:.2f}" for x in ms_one), flush=True)
    if plain:
        print("  plain table oxg_cut(0, 2) " + " ".join(f"{x:.1f}" for x in plain[0]) + f"; same count: {plain[1]}", flush=True)
        print("  plain table oxg_erase_hashes (host list) " + " ".join(f"{x:.1f}" for x in plain[2]) + f"; same count: {plain[3]}", flush=True)
for p in (d_b, d_o, d_q):
    capi.device_free(p, local)
dist.barrier()
dist.destroy_process_group()
