#!/usr/bin/env python
"""Point lookups on the sharded C3 table under torchrun (device-resident reads, as exp_shard.py).

Each rank asks QUERIES hashes (64 Mi) through oxg_shard_get_hashes_device: half present keys,
hashed from its own reads with hash_batch_device, half uniform random u64 (absent), shuffled.  A
call ends synchronised, so the wall time around it is the call's time; the max over ranks is what
a collective lookup of world * QUERIES hashes takes.  Prints G lookups/s per rank and in total, the
card name and power limit read in the same run, and at N=1 also the plain table's oxg_get_hashes
over host lists of the same hashes, for context.  Rank r runs on GPU r % (GPUs visible): with fewer GPUs
than ranks, shards share a device (and the exchange stays inside it; ranks that are separate processes on
one device time-slice it, so their rate is not a multi-GPU rate).  The launcher's own collectives are small
host-side ones, over gloo.

    torchrun --standalone --nproc-per-node N scripts/exp_shard_lookup.py
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
Q = int(os.environ.get("QUERIES", 64 << 20))
WARMUP, STEPS = 2, int(os.environ.get("STEPS", 5))
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

# the C3-shaped table: 12.5 M reads per rank, 1 % substitutions, 0.1 % N, genome 12.5 Mbp x N, k=21
d_b = capi.device_alloc(n * L + 64, local); d_o = capi.device_alloc((n + 1) * 8, local)
capi.synth_reads_device(d_b, n, L, G, 0xC30001, first_read=rank * n, sub_ppm=10_000, n_ppm=1_000, device=local)
capi.h2d(d_o, np.arange(n + 1, dtype=np.uint64) * np.uint64(L), local)
t = ShardedTable(k, rank, world, device=local, exchange=exchange)
t0 = time.perf_counter()
t.consume_batch_device(d_b, d_o, n, n * L, True)
build_s = mx(time.perf_counter() - t0)
size = t.stats()["len"]
slot_bytes = t.engine.table.capacity * 16

# queries: present keys from this rank's reads (windows across a read boundary or an N hash to 0:
# dropped), uniform random u64 for the other half
half = Q // 2
n_hr = min(n, half // (L - k + 1) * 5 // 4 + 1)
d_h = capi.device_alloc(n_hr * L * 8, local)
t.engine.table.hash_batch_device(d_b, d_o, n_hr, n_hr * L, d_h)
h = np.zeros(n_hr * L - k + 1, dtype=np.uint64)
capi.d2h(h, d_h, local)
capi.device_free(d_h, local)
present = h[h != 0][:half]
assert len(present) == half
rng = np.random.default_rng(1000 + rank)
order = rng.permutation(Q)
q = np.concatenate([present, rng.integers(0, (1 << 64) - 1, Q - half, dtype=np.uint64, endpoint=True)])[order]
is_present = order < half
d_q = capi.device_alloc(Q * 8, local); d_out = capi.device_alloc(Q * 8, local)
capi.h2d(d_q, q, local)


def timed(fn):
    ms = []
    for i in range(WARMUP + STEPS):
        dist.barrier()
        t0 = time.perf_counter()
        fn()
        wall = mx(time.perf_counter() - t0)
        if i >= WARMUP:
            ms.append(1e3 * wall)
    return ms


ms_dev = timed(lambda: t.engine.get_hashes_device(d_q, Q, d_out))
ans = np.zeros(Q, dtype=np.uint64)
capi.d2h(ans, d_out, local)
found_present = float(np.count_nonzero(ans[is_present])) / half
found_random = int(np.count_nonzero(ans[~is_present]))
ms_host = timed(lambda: t.engine.get_hashes(q))
same_host = bool(np.array_equal(t.engine.get_hashes(q), ans))
plain = None
if world == 1:
    # context: the shard's own table looked up directly (no routing), host lists in and out
    ms_plain = timed(lambda: t.engine.table.get_hashes(q))
    plain = (ms_plain, bool(np.array_equal(t.engine.table.get_hashes(q), ans)))
checks = [None] * world
dist.all_gather_object(checks, (found_present, found_random, same_host, size, slot_bytes))

if rank == 0:
    best = min(ms_dev)
    print(f"cards (rank: device, name, power limit): {cards}", flush=True)
    print(f"N={world}  C3-shaped table: {sum(c[3] for c in checks) / 1e9:.3f} G keys, "
          f"{[round(c[4] / 2**30, 1) for c in checks]} GiB of slots per shard, built in {build_s:.2f} s", flush=True)
    print(f"queries per rank {Q} (half present, half uniform random); ms per call, max over ranks:", flush=True)
    print("  get_hashes_device " + " ".join(f"{x:.1f}" for x in ms_dev)
          + f"  -> best {Q / best / 1e6:.2f} G lookups/s per rank, {world * Q / best / 1e6:.2f} G lookups/s in total", flush=True)
    print("  get_hashes (host lists) " + " ".join(f"{x:.1f}" for x in ms_host)
          + f"  -> best {Q / min(ms_host) / 1e6:.2f} G lookups/s per rank", flush=True)
    if plain:
        print("  plain table oxg_get_hashes (host lists, no routing) " + " ".join(f"{x:.1f}" for x in plain[0])
              + f"  -> best {Q / min(plain[0]) / 1e6:.2f} G lookups/s; same answers: {plain[1]}", flush=True)
    print(f"present keys found (per rank): {[c[0] for c in checks]}; random keys found: {[c[1] for c in checks]}; "
          f"host and device answers equal: {[c[2] for c in checks]}", flush=True)
for p in (d_b, d_o, d_q, d_out):
    capi.device_free(p, local)
dist.barrier()
t.close()
dist.destroy_process_group()
