"""Where the end-to-end step goes: wall clock of oxg_consume_batch on a pinned host batch against the
sum of its consume-kernel times, for several staging chunk sizes (set before the library loads)."""
import os, sys, time, numpy as np
sys.path.insert(0, '/root/repo')
from oxli_b200 import _capi as capi
n, L, k, G = 10_000_000, 150, 31, 5_000_000
d = capi.device_alloc(n * L + 64)
capi.synth_reads_device(d, n, L, G, 0xC20001)
h = capi.pinned_empty(n * L); capi.d2h(h, d); capi.device_free(d)
offs = np.arange(n + 1, dtype=np.uint64) * np.uint64(L)
t = capi.Table(k, capacity_hint=G)
for rep in range(4):
    t.clear()
    t0 = time.perf_counter(); st, total, _, _ = t.consume_batch(h, offs); dt = time.perf_counter() - t0
    ms, nl = t.last_consume_kernel_ms()
    print(f"chunk {os.environ.get('OXLI_B200_CHUNK_MB', '64')} MiB: wall {dt*1e3:.1f} ms, kernels {ms:.1f} ms in {nl} launches, {total/dt/1e9:.1f} G k-mers/s", flush=True)
# error mode = a pre-scan pass (same copies, kernels of ~0.2 ms per chunk) + the counting pass:
# the difference to the skip-mode wall time is what the copies cost when nothing competes
for rep in range(2):
    t.clear()
    t0 = time.perf_counter(); st, total, er, _ = t.consume_batch(h, offs, skip_bad=False); dt2 = time.perf_counter() - t0
    print(f"error mode (no bad k-mer, er={er}): wall {dt2*1e3:.1f} ms -> copy-only pass {dt2*1e3 - dt*1e3:.1f} ms = {n*L/(dt2-dt)/1e9:.1f} GB/s", flush=True)
