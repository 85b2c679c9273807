"""ctypes declarations for the C ABI in include/oxli_b200.h.

Thin, typed access to `liboxli_b200.so` for bench.py, the sharded driver and
the low-level tests (device-pointer entry points).  The drop-in
`KmerCountTable` class is the compiled module `oxli_b200._oxli`
(csrc/pyoxli.cpp); both sit on the same C ABI.  There is no fallback: a missing
library raises ImportError, a missing GPU makes every call raise OxliCudaError.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("OXLI_B200_LIB") or os.path.join(_HERE, "liboxli_b200.so")

OK, ERR_CUDA, ERR_INVALID, ERR_BAD_KMER, ERR_NOMEM, ERR_WRONG_KSIZE, ERR_TOO_SMALL, ERR_IO = range(8)

u64 = C.c_uint64
u64p = C.POINTER(C.c_uint64)
vp = C.c_void_p


class OxliError(RuntimeError):
    def __init__(self, status: int, msg: str):
        super().__init__(msg)
        self.status = status


class OxliCudaError(OxliError):
    pass


class OxliIOError(OxliError, OSError):
    """a file could not be created, opened or written (OXG_ERR_IO)"""


class oxg_stats(C.Structure):
    _fields_ = [("len", u64), ("sum", u64), ("min", u64), ("max", u64)]


# name -> (restype, argtypes).  Must list every symbol the header declares
# (tests/test_abi.py parses the header and checks).
SIGNATURES = {
    "oxg_last_error": (C.c_char_p, []),
    "oxg_version": (C.c_char_p, []),
    "oxg_device_count": (C.c_int, []),
    "oxg_table_create": (C.c_int, [C.c_int, C.c_uint32, u64, C.POINTER(vp)]),
    "oxg_table_destroy": (C.c_int, [vp]),
    "oxg_table_clear": (C.c_int, [vp]),
    "oxg_table_reserve": (C.c_int, [vp, u64]),
    "oxg_table_ksize": (C.c_int, [vp, C.POINTER(C.c_uint32)]),
    "oxg_table_capacity": (C.c_int, [vp, u64p]),
    "oxg_hash_windows": (C.c_int, [vp, vp, u64, vp]),
    "oxg_consume_batch": (C.c_int, [vp, vp, vp, u64, C.c_int, u64p, C.POINTER(C.c_int64), u64p]),
    "oxg_consume_batch_device": (C.c_int, [vp, vp, vp, u64, u64, C.c_int, u64p, C.POINTER(C.c_int64), u64p]),
    "oxg_hash_batch_device": (C.c_int, [vp, vp, vp, u64, u64, vp]),
    "oxg_count_hashes": (C.c_int, [vp, vp, u64, vp]),
    "oxg_count_hashes_device": (C.c_int, [vp, vp, u64, C.c_int, u64p]),
    "oxg_add_pairs": (C.c_int, [vp, vp, vp, u64]),
    "oxg_get_hashes": (C.c_int, [vp, vp, u64, vp]),
    "oxg_set_hash": (C.c_int, [vp, u64, u64]),
    "oxg_erase_hashes": (C.c_int, [vp, vp, u64, u64p]),
    "oxg_cut": (C.c_int, [vp, C.c_int, u64, u64p]),
    "oxg_table_len": (C.c_int, [vp, u64p]),
    "oxg_table_stats": (C.c_int, [vp, C.POINTER(oxg_stats)]),
    "oxg_histo": (C.c_int, [vp, vp, vp, u64, u64p]),
    "oxg_export": (C.c_int, [vp, vp, vp, u64, C.c_int, u64p]),
    "oxg_setop_sizes": (C.c_int, [vp, vp, u64p, u64p]),
    "oxg_setop_export": (C.c_int, [vp, vp, C.c_int, vp, u64, u64p]),
    "oxg_jaccard": (C.c_int, [vp, vp, C.POINTER(C.c_double)]),
    "oxg_cosine": (C.c_int, [vp, vp, C.POINTER(C.c_double)]),
    "oxg_merge": (C.c_int, [vp, vp, u64p, u64p]),
    "oxg_shard_create": (C.c_int, [C.c_int, C.c_uint32, C.c_int, C.c_int, u64, u64, C.POINTER(vp)]),
    "oxg_shard_destroy": (C.c_int, [vp]),
    "oxg_shard_table": (vp, [vp]),
    "oxg_shard_info": (C.c_int, [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_uint32), u64p, u64p]),
    "oxg_shard_export": (C.c_int, [vp, vp]),
    "oxg_shard_connect": (C.c_int, [vp, vp]),
    "oxg_shard_connect_local": (C.c_int, [C.POINTER(vp), C.c_int]),
    "oxg_shard_consume_batch": (C.c_int, [vp, vp, vp, u64, C.c_int, u64p, u64p, C.POINTER(C.c_int64), u64p]),
    "oxg_shard_consume_batch_device": (C.c_int, [vp, vp, vp, u64, u64, C.c_int, u64p, u64p, C.POINTER(C.c_int64), u64p]),
    "oxg_shard_get_hashes": (C.c_int, [vp, vp, u64, vp]),
    "oxg_shard_get_hashes_device": (C.c_int, [vp, vp, u64, vp]),
    "oxg_shard_merge_table": (C.c_int, [vp, vp, u64p, u64p]),
    "oxg_shard_merge": (C.c_int, [vp, vp, u64p, u64p]),
    "oxg_shard_erase_hashes": (C.c_int, [vp, vp, u64, u64p]),
    "oxg_shard_erase_hashes_device": (C.c_int, [vp, vp, u64, u64p]),
    "oxg_shard_cut": (C.c_int, [vp, C.c_int, u64, u64p]),
    "oxg_shard_export_pairs": (C.c_int, [vp, C.c_int, vp, vp, u64, u64p, vp, u64, u64p, u64p]),
    "oxg_shard_dump": (C.c_int, [vp, C.c_char_p, C.c_int]),
    "oxg_shard_last_ms": (C.c_int, [vp, C.POINTER(C.c_float), u64p]),
    "oxg_shard_stats": (C.c_int, [vp, C.POINTER(oxg_stats)]),
    "oxg_shard_histo": (C.c_int, [vp, vp, vp, u64, u64p]),
    "oxg_shard_setop_sizes": (C.c_int, [vp, vp, u64p, u64p]),
    "oxg_shard_jaccard": (C.c_int, [vp, vp, C.POINTER(C.c_double)]),
    "oxg_shard_digest": (C.c_int, [vp, vp]),
    "oxg_shard_allgather": (C.c_int, [vp, vp, C.c_uint32, vp]),
    "oxg_table_digest": (C.c_int, [vp, C.c_int, C.c_int, vp]),
    "oxg_synth_reads_device": (C.c_int, [C.c_int, vp, u64, C.c_uint32, u64, u64, u64, C.c_uint32, C.c_uint32]),
    "oxg_pinned_alloc": (C.c_int, [u64, C.POINTER(vp)]),
    "oxg_pinned_free": (C.c_int, [vp]),
    "oxg_device_alloc": (C.c_int, [C.c_int, u64, C.POINTER(vp)]),
    "oxg_device_free": (C.c_int, [C.c_int, vp]),
    "oxg_memcpy_h2d": (C.c_int, [C.c_int, vp, vp, u64]),
    "oxg_memcpy_d2h": (C.c_int, [C.c_int, vp, vp, u64]),
    "oxg_sync": (C.c_int, [vp]),
    "oxg_timer_start": (C.c_int, [vp]),
    "oxg_timer_stop": (C.c_int, [vp, C.POINTER(C.c_float)]),
    "oxg_launch_count": (u64, []),
    "oxg_live_allocations": (u64, []),
    "oxg_fail_allocation_after": (u64, [u64]),
    "oxg_last_consume_kernel_ms": (C.c_int, [vp, C.POINTER(C.c_float), u64p]),
    "oxg_set_pipeline": (C.c_int, [C.c_int, C.c_uint32, C.c_uint32]),
    "oxg_last_consume_pass_ms": (C.c_int, [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
}


def _load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m oxli_b200._build` "
            "(nvcc, sm_100a). oxli_b200 has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return lib


lib = _load()


def check(status: int) -> None:
    if status == OK:
        return
    msg = (lib.oxg_last_error() or b"").decode(errors="replace")
    if status == ERR_CUDA:
        raise OxliCudaError(status, msg)
    if status == ERR_IO:
        raise OxliIOError(status, msg)
    raise OxliError(status, msg)


def _ptr(a: np.ndarray | None):
    return None if a is None else a.ctypes.data


class Table:
    """Low-level handle wrapper (numpy in/out).  Not the drop-in class."""

    def __init__(self, ksize: int, device: int = 0, capacity_hint: int = 0):
        self._h = vp()
        check(lib.oxg_table_create(device, ksize, capacity_hint, C.byref(self._h)))
        self.ksize = ksize
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            lib.oxg_table_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def clear(self):
        check(lib.oxg_table_clear(self._h))

    def reserve(self, n):
        check(lib.oxg_table_reserve(self._h, n))

    @property
    def capacity(self) -> int:
        v = u64()
        check(lib.oxg_table_capacity(self._h, C.byref(v)))
        return int(v.value)

    def hash_windows(self, seq: bytes | np.ndarray) -> np.ndarray:
        a = np.frombuffer(seq, dtype=np.uint8) if not isinstance(seq, np.ndarray) else np.ascontiguousarray(seq, dtype=np.uint8)
        n = max(len(a) - self.ksize + 1, 0)
        out = np.zeros(n, dtype=np.uint64)
        if n:
            check(lib.oxg_hash_windows(self._h, a.ctypes.data, len(a), out.ctypes.data))
        return out

    def consume_batch(self, bases: np.ndarray, offsets: np.ndarray, skip_bad: bool = True):
        """Returns (status, total_counted, err_read, err_pos); status is OK or ERR_BAD_KMER."""
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        total, er, ep = u64(), C.c_int64(), u64()
        st = lib.oxg_consume_batch(self._h, _ptr(bases), _ptr(offsets), len(offsets) - 1, 1 if skip_bad else 0,
                                   C.byref(total), C.byref(er), C.byref(ep))
        if st not in (OK, ERR_BAD_KMER):
            check(st)
        return st, int(total.value), int(er.value), int(ep.value)

    def consume_batch_device(self, d_bases: int, d_offsets: int, n_reads: int, total_bases: int, skip_bad: bool = True):
        total, er, ep = u64(), C.c_int64(), u64()
        st = lib.oxg_consume_batch_device(self._h, d_bases, d_offsets, n_reads, total_bases, 1 if skip_bad else 0,
                                          C.byref(total), C.byref(er), C.byref(ep))
        if st not in (OK, ERR_BAD_KMER):
            check(st)
        return st, int(total.value), int(er.value), int(ep.value)

    def hash_batch_device(self, d_bases: int, d_offsets: int, n_reads: int, total_bases: int, d_out: int):
        check(lib.oxg_hash_batch_device(self._h, d_bases, d_offsets, n_reads, total_bases, d_out))

    def count_hashes(self, hashes, want_counts: bool = False):
        h = np.ascontiguousarray(hashes, dtype=np.uint64)
        out = np.empty(len(h), dtype=np.uint64) if want_counts else None
        check(lib.oxg_count_hashes(self._h, _ptr(h), len(h), _ptr(out)))
        return out

    def count_hashes_device(self, d_hashes: int, n: int, skip_zero: bool = False) -> int:
        c = u64()
        check(lib.oxg_count_hashes_device(self._h, d_hashes, n, 1 if skip_zero else 0, C.byref(c)))
        return int(c.value)

    def add_pairs(self, keys, vals):
        k = np.ascontiguousarray(keys, dtype=np.uint64)
        v = np.ascontiguousarray(vals, dtype=np.uint64)
        assert len(k) == len(v)
        check(lib.oxg_add_pairs(self._h, _ptr(k), _ptr(v), len(k)))

    def get_hashes(self, hashes) -> np.ndarray:
        h = np.ascontiguousarray(hashes, dtype=np.uint64)
        out = np.zeros(len(h), dtype=np.uint64)
        check(lib.oxg_get_hashes(self._h, _ptr(h), len(h), _ptr(out)))
        return out

    def set_hash(self, h: int, v: int):
        check(lib.oxg_set_hash(self._h, h, v))

    def erase_hashes(self, hashes) -> int:
        h = np.ascontiguousarray(hashes, dtype=np.uint64)
        n = u64()
        check(lib.oxg_erase_hashes(self._h, _ptr(h), len(h), C.byref(n)))
        return int(n.value)

    def cut(self, mode: int, thresh: int) -> int:
        n = u64()
        check(lib.oxg_cut(self._h, mode, thresh, C.byref(n)))
        return int(n.value)

    def __len__(self) -> int:
        n = u64()
        check(lib.oxg_table_len(self._h, C.byref(n)))
        return int(n.value)

    def stats(self) -> dict:
        s = oxg_stats()
        check(lib.oxg_table_stats(self._h, C.byref(s)))
        return {"len": int(s.len), "sum": int(s.sum), "min": int(s.min), "max": int(s.max)}

    def histo(self) -> list[tuple[int, int]]:
        n = u64()
        check(lib.oxg_histo(self._h, None, None, 0, C.byref(n)))
        f = np.zeros(max(int(n.value), 1), dtype=np.uint64)
        c = np.zeros(max(int(n.value), 1), dtype=np.uint64)
        check(lib.oxg_histo(self._h, _ptr(f), _ptr(c), len(f), C.byref(n)))
        return [(int(f[i]), int(c[i])) for i in range(int(n.value))]

    def export(self, sort_mode: int = 0) -> tuple[np.ndarray, np.ndarray]:
        n = u64()
        check(lib.oxg_export(self._h, None, None, 0, sort_mode, C.byref(n)))
        m = int(n.value)
        k = np.zeros(max(m, 1), dtype=np.uint64)
        v = np.zeros(max(m, 1), dtype=np.uint64)
        if m:
            check(lib.oxg_export(self._h, _ptr(k), _ptr(v), m, sort_mode, C.byref(n)))
        return k[:m], v[:m]

    def setop_sizes(self, other: "Table") -> tuple[int, int]:
        i, u = u64(), u64()
        check(lib.oxg_setop_sizes(self._h, other._h, C.byref(i), C.byref(u)))
        return int(i.value), int(u.value)

    def setop(self, other: "Table", op: int) -> np.ndarray:
        cap = len(self) + len(other) + 2
        out = np.zeros(cap, dtype=np.uint64)
        n = u64()
        check(lib.oxg_setop_export(self._h, other._h, op, _ptr(out), cap, C.byref(n)))
        return out[: int(n.value)]

    def jaccard(self, other: "Table") -> float:
        d = C.c_double()
        check(lib.oxg_jaccard(self._h, other._h, C.byref(d)))
        return float(d.value)

    def cosine(self, other: "Table") -> float:
        d = C.c_double()
        check(lib.oxg_cosine(self._h, other._h, C.byref(d)))
        return float(d.value)

    def merge(self, other: "Table") -> tuple[int, int]:
        a, n = u64(), u64()
        check(lib.oxg_merge(self._h, other._h, C.byref(a), C.byref(n)))
        return int(a.value), int(n.value)

    def sync(self):
        check(lib.oxg_sync(self._h))

    def timer_start(self):
        check(lib.oxg_timer_start(self._h))

    def timer_stop(self) -> float:
        ms = C.c_float()
        check(lib.oxg_timer_stop(self._h, C.byref(ms)))
        return float(ms.value)

    def last_consume_kernel_ms(self) -> tuple[float, int]:
        ms, n = C.c_float(), u64()
        check(lib.oxg_last_consume_kernel_ms(self._h, C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def last_consume_pass_ms(self) -> tuple[float, float]:
        a, b = C.c_float(), C.c_float()
        check(lib.oxg_last_consume_pass_ms(self._h, C.byref(a), C.byref(b)))
        return float(a.value), float(b.value)

    def device_digest(self, n_ranks: int = 1, rank: int = 0) -> dict:
        """The same digests computed by one scan on the device (oxg_table_digest)."""
        out = (u64 * 5)()
        check(lib.oxg_table_digest(self._h, n_ranks, rank, out))
        return {"n": int(out[0]), "sum": int(out[1]), "xor": int(out[2]), "sum_hc": int(out[3]), "foreign": int(out[4])}

    def digest(self) -> dict:
        """Order-independent digests of the (hash, count) multiset (test helper)."""
        k, v = self.export(1)
        with np.errstate(over="ignore"):
            return {
                "n": int(len(k)),
                "sum": int(v.sum(dtype=np.uint64)),
                "xor": int(np.bitwise_xor.reduce(k)) if len(k) else 0,
                "sum_hc": int((k * v).sum(dtype=np.uint64)),
            }


def set_pipeline(choice: int | str = 0, n_parts: int = 0, groups: int = 0) -> None:
    """0/'auto', 1/'fused', 2/'part' (see oxg_set_pipeline)."""
    choice = {"auto": 0, "fused": 1, "part": 2}.get(choice, choice)
    check(lib.oxg_set_pipeline(int(choice), n_parts, groups))


def device_alloc(nbytes: int, device: int = 0) -> int:
    p = vp()
    check(lib.oxg_device_alloc(device, nbytes, C.byref(p)))
    return int(p.value)


def device_free(ptr: int, device: int = 0) -> None:
    check(lib.oxg_device_free(device, ptr))


def h2d(d_dst: int, src: np.ndarray, device: int = 0) -> None:
    src = np.ascontiguousarray(src)
    check(lib.oxg_memcpy_h2d(device, d_dst, src.ctypes.data, src.nbytes))


def d2h(dst: np.ndarray, d_src: int, device: int = 0) -> None:
    check(lib.oxg_memcpy_d2h(device, dst.ctypes.data, d_src, dst.nbytes))


class Shard:
    """One shard of a hash-sharded table (low-level wrapper over oxg_shard_*).  Collective calls
    must be made by every rank; in one process, drive the ranks from one thread each."""

    def __init__(self, ksize: int, rank: int, n_ranks: int, device: int = 0, capacity_hint: int = 0,
                 round_windows: int = 0):
        self._h = vp()
        check(lib.oxg_shard_create(device, ksize, rank, n_ranks, capacity_hint, round_windows, C.byref(self._h)))
        self.ksize, self.rank, self.n_ranks, self.device = ksize, rank, n_ranks, device
        # the shard's own table through the plain table API (not owned: never destroyed from here)
        self.table = Table.__new__(Table)
        self.table._h = vp(lib.oxg_shard_table(self._h))
        self.table.ksize, self.table.device = ksize, device
        self.table.close = lambda: None

    def close(self):
        if getattr(self, "_h", None):
            lib.oxg_shard_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self) -> dict:
        r, n, p = C.c_int(), C.c_int(), C.c_uint32()
        w, e = u64(), u64()
        check(lib.oxg_shard_info(self._h, C.byref(r), C.byref(n), C.byref(p), C.byref(w), C.byref(e)))
        return {"rank": r.value, "n_ranks": n.value, "n_parts": p.value, "round_windows": w.value, "exchange_bytes": e.value}

    def export_handle(self) -> bytes:
        buf = (C.c_uint8 * 64)()
        check(lib.oxg_shard_export(self._h, buf))
        return bytes(buf)

    def connect(self, handles: list[bytes]):
        blob = b"".join(handles)
        assert len(blob) == 64 * self.n_ranks
        check(lib.oxg_shard_connect(self._h, C.c_char_p(blob)))

    @staticmethod
    def connect_local(shards: list["Shard"]):
        arr = (vp * len(shards))(*[s._h for s in shards])
        check(lib.oxg_shard_connect_local(arr, len(shards)))

    def consume_batch(self, bases: np.ndarray, offsets: np.ndarray, skip_bad: bool = True):
        """Returns (status, counted, absorbed, err_read, err_pos)."""
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        cn, ab, er, ep = u64(), u64(), C.c_int64(), u64()
        st = lib.oxg_shard_consume_batch(self._h, _ptr(bases), _ptr(offsets), len(offsets) - 1, 1 if skip_bad else 0,
                                         C.byref(cn), C.byref(ab), C.byref(er), C.byref(ep))
        if st not in (OK, ERR_BAD_KMER):
            check(st)
        return st, int(cn.value), int(ab.value), int(er.value), int(ep.value)

    def consume_batch_device(self, d_bases: int, d_offsets: int, n_reads: int, total_bases: int, skip_bad: bool = True):
        cn, ab, er, ep = u64(), u64(), C.c_int64(), u64()
        st = lib.oxg_shard_consume_batch_device(self._h, d_bases, d_offsets, n_reads, total_bases, 1 if skip_bad else 0,
                                                C.byref(cn), C.byref(ab), C.byref(er), C.byref(ep))
        if st not in (OK, ERR_BAD_KMER):
            check(st)
        return st, int(cn.value), int(ab.value), int(er.value), int(ep.value)

    def get_hashes(self, hashes) -> np.ndarray:
        """Counts of this rank's queries in the whole table (collective)."""
        h = np.ascontiguousarray(hashes, dtype=np.uint64)
        out = np.zeros(len(h), dtype=np.uint64)
        check(lib.oxg_shard_get_hashes(self._h, _ptr(h), len(h), _ptr(out)))
        return out

    def get_hashes_device(self, d_hashes: int, n: int, d_out: int) -> None:
        check(lib.oxg_shard_get_hashes_device(self._h, d_hashes, n, d_out))

    def merge_table(self, table: Table | None) -> tuple[int, int]:
        """Adds this rank's plain table (None: nothing) into the sharded table (collective).
        Returns (counts_added, new_keys) over the whole table."""
        a, n = u64(), u64()
        check(lib.oxg_shard_merge_table(self._h, None if table is None else table._h, C.byref(a), C.byref(n)))
        return int(a.value), int(n.value)

    def merge(self, other: "Shard") -> tuple[int, int]:
        """Adds the other sharded table's shard of this rank into this one (collective)."""
        a, n = u64(), u64()
        check(lib.oxg_shard_merge(self._h, other._h, C.byref(a), C.byref(n)))
        return int(a.value), int(n.value)

    def erase_hashes(self, hashes) -> int:
        """Removes this rank's keys from the whole table (collective).  Returns the distinct keys
        removed over the whole table."""
        h = np.ascontiguousarray(hashes, dtype=np.uint64)
        n = u64()
        check(lib.oxg_shard_erase_hashes(self._h, _ptr(h), len(h), C.byref(n)))
        return int(n.value)

    def erase_hashes_device(self, d_hashes: int, n: int) -> int:
        r = u64()
        check(lib.oxg_shard_erase_hashes_device(self._h, d_hashes, n, C.byref(r)))
        return int(r.value)

    def cut(self, mode: int, thresh: int) -> int:
        """mincut (mode 0) / maxcut (mode 1) on every shard (collective); keys removed in all."""
        n = u64()
        check(lib.oxg_shard_cut(self._h, mode, thresh, C.byref(n)))
        return int(n.value)

    def export_pairs(self, sort_mode: int = 0) -> tuple[np.ndarray, np.ndarray, np.ndarray, int]:
        """This rank's pairs in sort_mode order (0 slot, 1 key, 2 (count, key)), as oxg_export, with
        where they go in the whole table (collective): returns (keys, vals, runs, total), runs an
        (n_runs, 2) array of (global_start, length) covering keys / vals in order."""
        n, nr, tot = u64(), u64(), u64()
        check(lib.oxg_shard_export_pairs(self._h, sort_mode, None, None, 0, C.byref(n), None, 0, C.byref(nr), C.byref(tot)))
        k = np.zeros(max(n.value, 1), dtype=np.uint64)
        v = np.zeros(max(n.value, 1), dtype=np.uint64)
        runs = np.zeros((max(nr.value, 1), 2), dtype=np.uint64)
        # (collective: the sizing call above was one exchange, this is the second)
        check(lib.oxg_shard_export_pairs(self._h, sort_mode, _ptr(k), _ptr(v), len(k), C.byref(n), _ptr(runs), len(runs),
                                         C.byref(nr), C.byref(tot)))
        return k[: n.value], v[: n.value], runs[: nr.value], int(tot.value)

    def dump(self, path: str, sort_mode: int = 0) -> None:
        """The whole table into one file at `path`, the same path on every rank (collective)."""
        check(lib.oxg_shard_dump(self._h, os.fsencode(path), sort_mode))

    def last_ms(self) -> tuple[float, int]:
        ms, n = C.c_float(), u64()
        check(lib.oxg_shard_last_ms(self._h, C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def stats(self) -> dict:
        st = oxg_stats()
        check(lib.oxg_shard_stats(self._h, C.byref(st)))
        return {"len": st.len, "sum": st.sum, "min": st.min, "max": st.max}

    def histo(self) -> list[tuple[int, int]]:
        n = u64()
        check(lib.oxg_shard_histo(self._h, None, None, 0, C.byref(n)))
        f = np.empty(max(n.value, 1), dtype=np.uint64)
        m = np.empty(max(n.value, 1), dtype=np.uint64)
        # (collective: the sizing call above was one round, this is the second)
        check(lib.oxg_shard_histo(self._h, _ptr(f), _ptr(m), len(f), C.byref(n)))
        return [(int(a), int(b)) for a, b in zip(f[: n.value], m[: n.value])]

    def setop_sizes(self, other: "Shard") -> tuple[int, int]:
        i, u = u64(), u64()
        check(lib.oxg_shard_setop_sizes(self._h, other._h, C.byref(i), C.byref(u)))
        return int(i.value), int(u.value)

    def jaccard(self, other: "Shard") -> float:
        d = C.c_double()
        check(lib.oxg_shard_jaccard(self._h, other._h, C.byref(d)))
        return float(d.value)

    def digest(self) -> dict:
        out = (u64 * 5)()
        check(lib.oxg_shard_digest(self._h, out))
        return {"n": int(out[0]), "sum": int(out[1]), "xor": int(out[2]), "sum_hc": int(out[3]), "foreign": int(out[4])}

    def allgather(self, mine: bytes) -> list[bytes]:
        out = (C.c_uint8 * (len(mine) * self.n_ranks))()
        check(lib.oxg_shard_allgather(self._h, C.c_char_p(mine), len(mine), out))
        raw = bytes(out)
        return [raw[i * len(mine):(i + 1) * len(mine)] for i in range(self.n_ranks)]


def synth_reads_device(d_bases: int, n_reads: int, read_len: int, genome_len: int, seed: int,
                       first_read: int = 0, sub_ppm: int = 0, n_ppm: int = 0, device: int = 0) -> None:
    check(lib.oxg_synth_reads_device(device, d_bases, n_reads, read_len, genome_len, seed, first_read, sub_ppm, n_ppm))


def pinned_empty(nbytes: int) -> np.ndarray:
    """uint8 numpy view of freshly allocated pinned host memory (freed with the array)."""
    p = vp()
    check(lib.oxg_pinned_alloc(nbytes, C.byref(p)))
    buf = (C.c_uint8 * max(nbytes, 1)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=np.uint8, count=nbytes)
    _PINNED[arr.ctypes.data] = p.value
    return arr


_PINNED: dict[int, int] = {}


def pinned_free(arr: np.ndarray) -> None:
    p = _PINNED.pop(arr.ctypes.data, None)
    if p:
        lib.oxg_pinned_free(p)
