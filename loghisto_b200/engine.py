"""Thin object wrapper over the C ABI (include/loghisto_b200.h).

`Engine` is what the host-side MetricSystem mirror, the tests and bench.py
drive.  It adds no arithmetic of its own: every bucket, count and percentile
comes out of the CUDA kernels behind `lh_*`.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib as L


class LhError(RuntimeError):
    def __init__(self, status: int, detail: str = ""):
        self.status = status
        msg = L.load().lh_strerror(status).decode()
        super().__init__(f"loghisto_b200: {msg} ({status})" + (f": {detail}" if detail else ""))


def _ptr(x) -> int:
    """Raw address of a device/host buffer: int, DeviceArray, torch tensor, numpy array or CAI object."""
    if x is None:
        return 0
    if isinstance(x, int):
        return x
    if isinstance(x, DeviceArray):
        return x.ptr
    if isinstance(x, np.ndarray):
        return x.ctypes.data
    if hasattr(x, "data_ptr"):
        return int(x.data_ptr())
    if hasattr(x, "__cuda_array_interface__"):
        return int(x.__cuda_array_interface__["data"][0])
    raise TypeError(f"cannot take the address of {type(x)!r}")


def _stream(s) -> int:
    if s is None:
        return 0
    if isinstance(s, int):
        return s
    if hasattr(s, "cuda_stream"):   # torch.cuda.Stream
        return int(s.cuda_stream)
    raise TypeError(f"not a stream: {type(s)!r}")


class DeviceArray:
    """Device memory owned through lh_device_alloc; exposes __cuda_array_interface__."""

    def __init__(self, engine: "Engine", n: int, dtype):
        self.engine = engine
        self.dtype = np.dtype(dtype)
        self.n = int(n)
        self.nbytes = self.n * self.dtype.itemsize
        p = C.c_void_p()
        engine._check(engine.lib.lh_device_alloc(engine.h, max(self.nbytes, 1), C.byref(p)))
        self.ptr = int(p.value)

    @property
    def __cuda_array_interface__(self):
        return {"shape": (self.n,), "typestr": self.dtype.str, "data": (self.ptr, False), "version": 3}

    def offset(self, elems: int) -> int:
        return self.ptr + elems * self.dtype.itemsize

    def to_host(self) -> np.ndarray:
        out = np.empty(self.n, dtype=self.dtype)
        if self.nbytes:
            self.engine._check(self.engine.lib.lh_memcpy_d2h(self.engine.h, out.ctypes.data, self.ptr, self.nbytes))
        return out

    def free(self):
        if self.ptr and self.engine.h:
            self.engine.lib.lh_device_free(self.engine.h, self.ptr)
        self.ptr = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class PinnedArray:
    """Pinned host memory from lh_host_alloc_pinned, viewed as a numpy array."""

    def __init__(self, engine: "Engine", n: int, dtype):
        self.engine = engine
        self.dtype = np.dtype(dtype)
        self.n = int(n)
        self.nbytes = self.n * self.dtype.itemsize
        p = C.c_void_p()
        engine._check(engine.lib.lh_host_alloc_pinned(engine.h, max(self.nbytes, 1), C.byref(p)))
        self.ptr = int(p.value)
        buf = (C.c_char * max(self.nbytes, 1)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=self.n)

    def free(self):
        if self.ptr and self.engine.h:
            self.array = None
            self.engine.lib.lh_host_free_pinned(self.engine.h, self.ptr)
        self.ptr = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


@dataclass
class Reduced:
    counts: np.ndarray   # uint64[H]
    sums: np.ndarray     # float64[H]
    avgs: np.ndarray     # float64[H]
    pkeys: np.ndarray    # int32[H, np]  (INT32_MIN = percentile() error)
    pvals: np.ndarray    # float64[H, np]


@dataclass
class Sparse:
    offsets: np.ndarray        # uint32[H+1]
    keys: np.ndarray           # int16[total]
    counts: np.ndarray         # uint64[total]
    counter_deltas: np.ndarray  # uint64[C]

    def histogram(self, hid: int) -> dict:
        a, b = int(self.offsets[hid]), int(self.offsets[hid + 1])
        return {int(k): int(c) for k, c in zip(self.keys[a:b], self.counts[a:b])}


class Engine:
    def __init__(self, device: int = 0, max_histograms: int = 1, max_counters: int = 1,
                 staging_bytes: int = 0, staging_slots: int = 0, precision: int = 0):
        self.lib = L.load()
        self.h = None
        cfg = L.lh_config(C.sizeof(L.lh_config), device, max_histograms, max_counters,
                          staging_bytes, staging_slots, 0, precision)
        h = C.c_void_p()
        st = self.lib.lh_create(C.byref(cfg), C.byref(h))
        if st != L.LH_OK:
            raise LhError(st, "lh_create")
        self.h = h
        self.device = device
        self.H = max_histograms
        self.C = max_counters

    # ---- plumbing
    def _check(self, st: int):
        if st != L.LH_OK:
            raise LhError(st, self.lib.lh_last_error(self.h).decode() if self.h else "")

    def close(self):
        if self.h:
            self.lib.lh_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def alloc(self, n: int, dtype) -> DeviceArray:
        return DeviceArray(self, n, dtype)

    def pinned(self, n: int, dtype) -> PinnedArray:
        return PinnedArray(self, n, dtype)

    def upload(self, arr: np.ndarray) -> DeviceArray:
        arr = np.ascontiguousarray(arr)
        d = DeviceArray(self, arr.size, arr.dtype)
        if arr.nbytes:
            self._check(self.lib.lh_memcpy_h2d(self.h, d.ptr, arr.ctypes.data, arr.nbytes))
        return d

    def sync(self):
        self._check(self.lib.lh_sync(self.h))

    @property
    def ingest_stream(self) -> int:
        return int(self.lib.lh_ingest_stream(self.h) or 0)

    def tune(self, key: str, value: int):
        self._check(self.lib.lh_tune(self.h, key.encode(), int(value)))

    def k1_variants(self) -> list:
        return [self.lib.lh_k1_variant_name(self.h, i).decode() for i in range(self.lib.lh_k1_variant_count())]

    def k1_variant_name(self) -> str:
        return self.lib.lh_k1_variant_name(self.h, self.lib.lh_k1_variant_current(self.h)).decode()

    def keyed_kernel_name(self) -> str:
        """Name of the kernel the most recent keyed ingest dispatched to."""
        return self.lib.lh_keyed_kernel_name(self.h).decode()

    # ---- multi-GPU (peer-memory all-reduce behind the ABI)
    def comm_export(self) -> bytes:
        buf = C.create_string_buffer(L.LH_PEER_HANDLE_BYTES)
        self._check(self.lib.lh_comm_export(self.h, buf))
        return buf.raw

    def comm_import(self, rank: int, world: int, handles: bytes):
        assert len(handles) == world * L.LH_PEER_HANDLE_BYTES
        self._check(self.lib.lh_comm_import(self.h, rank, world, C.c_char_p(handles)))

    def snapshot_allreduce(self, counters: bool = False) -> int:
        seq = C.c_uint64()
        self._check(self.lib.lh_snapshot_allreduce(self.h, 1 if counters else 0, C.byref(seq)))
        return int(seq.value)

    def comm_allreduce_ms(self, seq: int) -> float:
        ms = C.c_float()
        self._check(self.lib.lh_comm_allreduce_ms(self.h, seq, C.byref(ms)))
        return float(ms.value)

    def comm_info(self) -> dict:
        st = L.lh_comm_stats()
        self._check(self.lib.lh_comm_info(self.h, C.byref(st)))
        return {f: int(getattr(st, f)) for f, _ in L.lh_comm_stats._fields_ if f != "reserved"}

    def comm_last_bytes(self) -> int:
        return self.comm_info()["last_bytes_from_peers"]

    def last_kernel_ms(self) -> float:
        ms = C.c_float()
        self._check(self.lib.lh_last_kernel_ms(self.h, C.byref(ms)))
        return float(ms.value)

    def ingest_seq(self) -> int:
        return int(self.lib.lh_ingest_seq(self.h))

    def kernel_ms(self, seq: int) -> float:
        ms = C.c_float()
        self._check(self.lib.lh_kernel_ms(self.h, seq, C.byref(ms)))
        return float(ms.value)

    def stats(self) -> dict:
        s = L.lh_stats()
        self._check(self.lib.lh_get_stats(self.h, C.byref(s)))
        return {f: int(getattr(s, f)) for f, _ in L.lh_stats._fields_}

    # ---- ingest, device inputs
    def ingest_f64(self, histogram_id: int, d_values, n: int, stream=None):
        self._check(self.lib.lh_ingest_f64(self.h, histogram_id, _ptr(d_values), n, _stream(stream)))

    def ingest_keyed_f64_u16(self, d_ids, d_values, n: int, stream=None):
        self._check(self.lib.lh_ingest_keyed_f64_u16(self.h, _ptr(d_ids), _ptr(d_values), n, _stream(stream)))

    def ingest_keyed_f64_u32(self, d_ids, d_values, n: int, stream=None):
        self._check(self.lib.lh_ingest_keyed_f64_u32(self.h, _ptr(d_ids), _ptr(d_values), n, _stream(stream)))

    def ingest_keyed_i64ns_u16(self, d_ids, d_nanos, n: int, stream=None):
        self._check(self.lib.lh_ingest_keyed_i64ns_u16(self.h, _ptr(d_ids), _ptr(d_nanos), n, _stream(stream)))

    def ingest_keyed_pair_u16(self, d_ids_f64, d_values, n_f64: int, d_ids_ns, d_nanos, n_ns: int, stream=None):
        """Histogram samples and Timer samples of one batch in one call (one launch of the write-combining kernel)."""
        self._check(self.lib.lh_ingest_keyed_pair_u16(self.h, _ptr(d_ids_f64), _ptr(d_values), n_f64, _ptr(d_ids_ns), _ptr(d_nanos), n_ns,
                                                      _stream(stream)))

    def counter_add_u16(self, d_ids, d_amounts, n: int, stream=None):
        self._check(self.lib.lh_counter_add_u16(self.h, _ptr(d_ids), _ptr(d_amounts), n, _stream(stream)))

    def counter_add_u32(self, d_ids, d_amounts, n: int, stream=None):
        self._check(self.lib.lh_counter_add_u32(self.h, _ptr(d_ids), _ptr(d_amounts), n, _stream(stream)))

    # ---- ingest, host inputs
    def ingest_f64_host(self, histogram_id: int, h_values, n: int | None = None):
        if isinstance(h_values, np.ndarray):
            assert h_values.dtype == np.float64 and h_values.flags.c_contiguous
            n = h_values.size if n is None else n
        self._check(self.lib.lh_ingest_f64_host(self.h, histogram_id, _ptr(h_values), n))

    def ingest_keyed_f64_u16_host(self, h_ids, h_values, n: int | None = None):
        if isinstance(h_values, np.ndarray):
            assert h_values.dtype == np.float64 and h_ids.dtype == np.uint16
            n = h_values.size if n is None else n
        self._check(self.lib.lh_ingest_keyed_f64_u16_host(self.h, _ptr(h_ids), _ptr(h_values), n))

    def ingest_keyed_i64ns_u16_host(self, h_ids, h_nanos, n: int | None = None):
        if isinstance(h_nanos, np.ndarray):
            assert h_nanos.dtype == np.int64 and h_ids.dtype == np.uint16
            n = h_nanos.size if n is None else n
        self._check(self.lib.lh_ingest_keyed_i64ns_u16_host(self.h, _ptr(h_ids), _ptr(h_nanos), n))

    def counter_add_u16_host(self, h_ids, h_amounts, n: int | None = None):
        if isinstance(h_amounts, np.ndarray):
            assert h_amounts.dtype == np.uint64 and h_ids.dtype == np.uint16
            n = h_amounts.size if n is None else n
        self._check(self.lib.lh_counter_add_u16_host(self.h, _ptr(h_ids), _ptr(h_amounts), n))

    def merge_counts_host(self, ids, keys, counts):
        """Add sparse (histogram id, int16 key, uint64 count) triples into the active arrays (exact merge)."""
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        keys = np.ascontiguousarray(keys, dtype=np.int16)
        counts = np.ascontiguousarray(counts, dtype=np.uint64)
        assert ids.size == keys.size == counts.size
        self._check(self.lib.lh_merge_counts_host(self.h, ids.ctypes.data, keys.ctypes.data, counts.ctypes.data, ids.size))

    # ---- staging ring
    def staging_acquire(self) -> L.lh_staging:
        s = L.lh_staging()
        self._check(self.lib.lh_staging_acquire(self.h, C.byref(s)))
        return s

    def staging_view(self, s: L.lh_staging, dtype, count: int, byte_offset: int = 0) -> np.ndarray:
        buf = (C.c_char * int(s.bytes)).from_address(s.host)
        return np.frombuffer(buf, dtype=dtype, count=count, offset=byte_offset)

    def staging_commit_f64(self, s, histogram_id: int, n: int):
        self._check(self.lib.lh_staging_commit_f64(self.h, C.byref(s), histogram_id, n))

    def staging_commit_keyed_f64_u16(self, s, n: int, ids_offset: int):
        self._check(self.lib.lh_staging_commit_keyed_f64_u16(self.h, C.byref(s), n, ids_offset))

    def staging_commit_counter_u16(self, s, n: int, ids_offset: int):
        self._check(self.lib.lh_staging_commit_counter_u16(self.h, C.byref(s), n, ids_offset))

    def staging_abandon(self, s):
        self._check(self.lib.lh_staging_abandon(self.h, C.byref(s)))

    # ---- snapshot
    def snapshot_begin(self):
        self._check(self.lib.lh_snapshot_begin(self.h))

    def snapshot_device(self) -> L.lh_device_view:
        v = L.lh_device_view()
        self._check(self.lib.lh_snapshot_device(self.h, C.byref(v)))
        return v

    def _reduce_into(self, fn, percentiles) -> Reduced:
        """fn(ctx, ps, np, counts, sums, avgs, pkeys, pvals): lh_snapshot_reduce or lh_window_reduce."""
        ps = np.ascontiguousarray(percentiles, dtype=np.float64)
        npct = ps.size
        H = self.H
        counts = np.zeros(H, dtype=np.uint64)
        sums = np.zeros(H, dtype=np.float64)
        avgs = np.zeros(H, dtype=np.float64)
        pkeys = np.zeros((H, npct), dtype=np.int32)
        pvals = np.zeros((H, npct), dtype=np.float64)
        self._check(fn(self.h, ps.ctypes.data if npct else 0, npct, counts.ctypes.data, sums.ctypes.data,
                       avgs.ctypes.data, pkeys.ctypes.data, pvals.ctypes.data))
        return Reduced(counts, sums, avgs, pkeys, pvals)

    def snapshot_reduce(self, percentiles) -> Reduced:
        return self._reduce_into(self.lib.lh_snapshot_reduce, percentiles)

    def snapshot_reduce_async(self, percentiles) -> tuple:
        """Enqueue the reduction; returns an opaque handle for snapshot_result()."""
        ps = np.ascontiguousarray(percentiles, dtype=np.float64)
        t = C.c_uint64()
        self._check(self.lib.lh_snapshot_reduce_async(self.h, ps.ctypes.data if ps.size else 0, ps.size, C.byref(t)))
        return (int(t.value), ps.size)

    def snapshot_result(self, handle) -> Reduced:
        ticket, npct = handle
        H = self.H
        counts = np.zeros(H, dtype=np.uint64)
        sums = np.zeros(H, dtype=np.float64)
        avgs = np.zeros(H, dtype=np.float64)
        pkeys = np.zeros((H, npct), dtype=np.int32)
        pvals = np.zeros((H, npct), dtype=np.float64)
        self._check(self.lib.lh_snapshot_result(self.h, ticket, counts.ctypes.data, sums.ctypes.data, avgs.ctypes.data,
                                                pkeys.ctypes.data, pvals.ctypes.data))
        return Reduced(counts, sums, avgs, pkeys, pvals)

    def _export_from(self, fn) -> Sparse:
        """fn(ctx, lh_sparse *): lh_snapshot_export or lh_window_export; the lists are copied out of the library's buffers."""
        sp = L.lh_sparse()
        self._check(fn(self.h, C.byref(sp)))
        total = int(sp.total_entries)
        offsets = np.ctypeslib.as_array(sp.offsets, shape=(self.H + 1,)).copy()
        keys = np.ctypeslib.as_array(sp.keys, shape=(total,)).copy() if total else np.zeros(0, np.int16)
        counts = np.ctypeslib.as_array(sp.counts, shape=(total,)).copy() if total else np.zeros(0, np.uint64)
        deltas = np.ctypeslib.as_array(sp.counter_deltas, shape=(self.C,)).copy()
        return Sparse(offsets, keys, counts, deltas)

    def snapshot_export(self) -> Sparse:
        return self._export_from(self.lib.lh_snapshot_export)

    def snapshot_copy_histogram(self, histogram_id: int) -> np.ndarray:
        out = np.zeros(65536, dtype=np.uint64)
        self._check(self.lib.lh_snapshot_copy_histogram(self.h, histogram_id, out.ctypes.data))
        return out

    def snapshot_end(self):
        self._check(self.lib.lh_snapshot_end(self.h))

    def snapshot(self, percentiles, export: bool = True):
        """begin + reduce (+ export) + end; returns (Reduced, Sparse | None)."""
        self.snapshot_begin()
        try:
            red = self.snapshot_reduce(percentiles)
            sp = self.snapshot_export() if export else None
        finally:
            self.snapshot_end()
        return red, sp

    # ---- windows: sums over the last K folded snapshots (K = 0: every snapshot since configure), on the device
    def window_configure(self, intervals: int):
        self._check(self.lib.lh_window_configure(self.h, intervals))

    def window_release(self):
        self._check(self.lib.lh_window_release(self.h))

    def window_fold(self):
        """Fold the open snapshot (after any all-reduce) into the window; once per snapshot."""
        self._check(self.lib.lh_window_fold(self.h))

    def window_reduce(self, percentiles) -> Reduced:
        return self._reduce_into(self.lib.lh_window_reduce, percentiles)

    def window_export(self) -> Sparse:
        return self._export_from(self.lib.lh_window_export)

    def window_info(self) -> dict:
        st = L.lh_window_stats()
        self._check(self.lib.lh_window_info(self.h, C.byref(st)))
        return {f: int(getattr(st, f)) for f, _ in L.lh_window_stats._fields_}

    # ---- probes / streams
    def compress(self, values: np.ndarray, mode: int = 0) -> np.ndarray:
        values = np.ascontiguousarray(values, dtype=np.float64)
        d_in = self.upload(values)
        d_out = self.alloc(values.size, np.int16)
        self._check(self.lib.lh_compress_f64(self.h, d_in.ptr, values.size, d_out.ptr, mode, 0))
        self.sync()
        out = d_out.to_host()
        d_in.free()
        d_out.free()
        return out

    def decompress_table(self) -> np.ndarray:
        out = np.zeros(65536, dtype=np.float64)
        self._check(self.lib.lh_decompress_table(self.h, out.ctypes.data))
        return out

    def fastpath_margin(self, d_values, n: int):
        err = C.c_double()
        slow = C.c_uint64()
        self._check(self.lib.lh_fastpath_margin(self.h, _ptr(d_values), n, C.byref(err), C.byref(slow), 0))
        return float(err.value), int(slow.value)

    def fastpath_margin_detail(self):
        a, b = C.c_double(), C.c_double()
        self._check(self.lib.lh_fastpath_margin_detail(self.h, C.byref(a), C.byref(b)))
        return float(a.value), float(b.value)

    def gen_stream(self, kind: int, n: int, seed: int, start: int = 0, out: DeviceArray | None = None,
                   stream=None) -> DeviceArray:
        if out is None:
            out = self.alloc(n, np.float64)
        self._check(self.lib.lh_gen_stream_f64(self.h, kind, seed, start, n, out.ptr, _stream(stream)))
        return out

    def gen_ids_u16(self, kind: int, n: int, n_ids: int, seed: int, start: int = 0,
                    out: DeviceArray | None = None, stream=None) -> DeviceArray:
        if out is None:
            out = self.alloc(n, np.uint16)
        self._check(self.lib.lh_gen_ids_u16(self.h, kind, seed, start, n, n_ids, out.ptr, _stream(stream)))
        return out
