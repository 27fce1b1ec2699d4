"""ctypes binding of librsp_b200.so (include/rsp_b200.h): the product's Python face.

There is no CPU path behind these classes: if the CUDA library is missing or no B200 is visible the
constructors raise.  Method names on `Shard` follow the reference's rocksdb::DB / DbWrapper usage
(rocksdb_replicator/rocksdb_wrapper.cpp, rocksdb_admin/application_db.cpp).
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(HERE, "librsp_b200.so")

OK, NOT_FOUND, CORRUPTION, NOT_SUPPORTED, INVALID_ARGUMENT, IO_ERROR = 0, 1, 2, 3, 4, 5
INCOMPLETE = 7
MERGE_NONE, MERGE_COUNTER, MERGE_UINT64ADD, MERGE_APPEND, MERGE_CALLBACK = 0, 1, 2, 3, 4

MERGE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p,
                       C.c_size_t, C.c_void_p, C.c_void_p)


class EngineCfg(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("max_shards", C.c_uint32), ("arena_bytes", C.c_uint64),
                ("staging_bytes", C.c_uint64), ("l0_compaction_trigger", C.c_uint32), ("reserved", C.c_uint32)]


class ShardOpts(C.Structure):
    _fields_ = [("merge_op", C.c_uint32), ("reserved", C.c_uint32), ("write_buffer_bytes", C.c_uint64),
                ("merge_fn", C.c_void_p), ("merge_state", C.c_void_p)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "latest_seq", "memtable_entries", "memtable_bytes", "n_runs", "run_entries", "run_bytes", "flushes",
        "compactions", "compaction_bytes_read", "compaction_bytes_written", "flush_comparison_sorts")]


EXPORTS = {
    # name: (restype, argtypes)
    "rsp_version": (C.c_char_p, []),
    "rsp_engine_create": (C.c_int, [C.c_int, C.POINTER(EngineCfg), C.POINTER(C.c_void_p)]),
    "rsp_engine_destroy": (None, [C.c_void_p]),
    "rsp_engine_device": (C.c_int, [C.c_void_p]),
    "rsp_engine_stream": (C.c_void_p, [C.c_void_p]),
    "rsp_shard_open": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(ShardOpts), C.POINTER(C.c_void_p)]),
    "rsp_shard_close": (C.c_int, [C.c_void_p]),
    "rsp_shard_index": (C.c_uint32, [C.c_void_p]),
    "rsp_shard_name": (C.c_char_p, [C.c_void_p]),
    "rsp_apply": (C.c_int, [C.c_void_p, C.c_char_p, C.c_size_t, C.c_uint64, C.POINTER(C.c_uint64)]),
    "rsp_write": (C.c_int, [C.c_void_p, C.c_char_p, C.c_size_t, C.POINTER(C.c_uint64)]),
    "rsp_apply_many": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p]),
    "rsp_apply_updates": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.POINTER(C.c_size_t)]),
    "rsp_multi_get_slices": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "rsp_router_create": (C.c_int, [C.c_size_t, C.c_void_p, C.POINTER(C.c_void_p)]),
    "rsp_router_destroy": (None, [C.c_void_p]),
    "rsp_router_add_shard": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p]),
    "rsp_router_remove_shard": (C.c_int, [C.c_void_p, C.c_uint32]),
    "rsp_router_multi_get": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_size_t, C.c_void_p, C.c_void_p]),
    "rsp_router_multi_get_fixed": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                             C.c_size_t, C.c_void_p, C.c_void_p]),
    "rsp_router_apply_many": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p]),
    "rsp_latest_seq": (C.c_uint64, [C.c_void_p]),
    "rsp_set_latest_seq": (C.c_int, [C.c_void_p, C.c_uint64]),
    "rsp_last_error": (C.c_size_t, [C.c_void_p, C.c_char_p, C.c_size_t]),
    "rsp_get": (C.c_int, [C.c_void_p, C.c_char_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "rsp_multi_get": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_size_t, C.c_void_p, C.c_void_p]),
    "rsp_multi_get_fixed": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                      C.c_size_t, C.c_void_p, C.c_void_p]),
    "rsp_iter_create": (C.c_void_p, [C.c_void_p]),
    "rsp_iter_destroy": (None, [C.c_void_p]),
    "rsp_iter_seek_to_first": (None, [C.c_void_p]),
    "rsp_iter_seek_to_last": (None, [C.c_void_p]),
    "rsp_iter_seek": (None, [C.c_void_p, C.c_char_p, C.c_size_t]),
    "rsp_iter_next": (None, [C.c_void_p]),
    "rsp_iter_prev": (None, [C.c_void_p]),
    "rsp_iter_valid": (C.c_int, [C.c_void_p]),
    "rsp_iter_key": (C.c_void_p, [C.c_void_p, C.POINTER(C.c_size_t)]),
    "rsp_iter_value": (C.c_void_p, [C.c_void_p, C.POINTER(C.c_size_t)]),
    "rsp_iter_status": (C.c_int, [C.c_void_p]),
    "rsp_multi_scan": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                 C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "rsp_flush": (C.c_int, [C.c_void_p]),
    "rsp_compact": (C.c_int, [C.c_void_p]),
    "rsp_flush_all": (C.c_int, [C.c_void_p]),
    "rsp_compact_all": (C.c_int, [C.c_void_p]),
    "rsp_get_stats": (C.c_int, [C.c_void_p, C.POINTER(Stats)]),
    "rsp_ingest_sorted": (C.c_int, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_void_p, C.c_char_p, C.c_void_p, C.c_int,
                                    C.POINTER(C.c_uint64)]),
    "rsp_multi_get_device": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                                       C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rsp_multi_scan_device": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                                        C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rsp_stage_build": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.POINTER(C.c_void_p)]),
    "rsp_stage_free": (None, [C.c_void_p]),
    "rsp_reserve": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rsp_apply_staged_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "rsp_apply_staged_finish": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "rsp_last_kernel_ms": (C.c_float, [C.c_void_p, C.c_char_p]),
    "rsp_kernel_launches": (C.c_uint64, [C.c_void_p]),
    "rsp_debug_last_pending": (C.c_uint32, [C.c_void_p, C.c_void_p, C.c_uint32]),
    "rsp_debug_combiner_stats": (None, [C.c_void_p, C.c_int, C.c_void_p]),
    "rsp_debug_arena": (None, [C.c_void_p, C.c_void_p]),
    "rsp_debug_run": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
}

_lib = None


def load_library():
    """dlopen librsp_b200.so and bind every symbol include/rsp_b200.h declares.  No compute."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise RuntimeError(
            f"{SO_PATH} is missing: build it with `python -m rocksplicator_b200.build` "
            "(the engine has no CPU fallback)")
    lib = C.CDLL(SO_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)  # AttributeError == a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class Iterator:
    def __init__(self, shard):
        self.lib = shard.lib
        self.h = self.lib.rsp_iter_create(shard.h)
        self._shard = shard

    def close(self):
        if self.h:
            self.lib.rsp_iter_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def seek_to_first(self): self.lib.rsp_iter_seek_to_first(self.h)
    def seek_to_last(self): self.lib.rsp_iter_seek_to_last(self.h)
    def seek(self, k): self.lib.rsp_iter_seek(self.h, k, len(k))
    def next(self): self.lib.rsp_iter_next(self.h)
    def prev(self): self.lib.rsp_iter_prev(self.h)
    def valid(self): return bool(self.lib.rsp_iter_valid(self.h))
    def status(self): return self.lib.rsp_iter_status(self.h)

    def key(self):
        n = C.c_size_t()
        p = self.lib.rsp_iter_key(self.h, C.byref(n))
        return C.string_at(p, n.value) if n.value else b""

    def value(self):
        n = C.c_size_t()
        p = self.lib.rsp_iter_value(self.h, C.byref(n))
        return C.string_at(p, n.value) if n.value else b""


class Shard:
    """One DB ("segment%05d"): apply == DbWrapper::HandleReplicateResponse, write == WriteToLeader,
    latest_seq == LatestSequenceNumber, get/multi_get/iterator == the ApplicationDB read surface."""

    def __init__(self, engine, name, merge_op=MERGE_NONE, write_buffer_bytes=0, merge_fn=None):
        self.engine = engine
        self.lib = engine.lib
        self.kind = "b200"
        opts = ShardOpts(merge_op=merge_op, write_buffer_bytes=write_buffer_bytes)
        self._merge_fn = None
        if merge_fn is not None:
            self._merge_fn = MERGE_FN(merge_fn)
            opts.merge_fn = C.cast(self._merge_fn, C.c_void_p)
        h = C.c_void_p()
        rc = self.lib.rsp_shard_open(engine.h, name.encode(), C.byref(opts), C.byref(h))
        if rc != OK:
            raise RuntimeError(f"rsp_shard_open({name}) -> {rc}")
        self.h = h
        self.name = name
        self.index = self.lib.rsp_shard_index(h)

    def close(self):
        if self.h:
            self.lib.rsp_shard_close(self.h)
            self.h = None

    @property
    def last_error(self):
        buf = C.create_string_buffer(256)
        self.lib.rsp_last_error(self.h, buf, 256)
        return buf.value.decode()

    def apply(self, batch: bytes, ts_ms: int = 0) -> int:
        return self.lib.rsp_apply(self.h, batch, len(batch), ts_ms, None)

    def write(self, batch: bytes) -> int:
        return self.lib.rsp_write(self.h, batch, len(batch), None)

    def latest_seq(self) -> int:
        return self.lib.rsp_latest_seq(self.h)

    def get(self, key: bytes, cap: int = 256):
        while True:
            buf = C.create_string_buffer(max(cap, 1))
            n = C.c_size_t()
            rc = self.lib.rsp_get(self.h, key, len(key), buf, cap, C.byref(n))
            if rc == INCOMPLETE:
                cap = n.value
                continue
            return (rc, buf.raw[:n.value]) if rc == OK else (rc, None)

    def multi_get(self, keys, stride=256):
        res = self.engine.multi_get([self.index] * len(keys), keys, stride)
        return res

    def iterator(self):
        return Iterator(self)

    def scan(self, start=None, limit=None):
        it = self.iterator()
        if start is None:
            it.seek_to_first()
        else:
            it.seek(start)
        out = []
        while it.valid() and (limit is None or len(out) < limit):
            out.append((it.key(), it.value()))
            it.next()
        it.close()
        return out

    def flush(self): return self.lib.rsp_flush(self.h)
    def compact(self): return self.lib.rsp_compact(self.h)

    def ingest(self, sorted_kv, allow_global_seqno=True) -> int:
        """DB::IngestExternalFile for sorted (key, value) pairs (see rocksplicator_b200/sst.py for SST files)"""
        n = len(sorted_kv)
        koff = np.zeros(n + 1, dtype=np.uint64)
        voff = np.zeros(n + 1, dtype=np.uint64)
        np.cumsum(np.fromiter((len(k) for k, _ in sorted_kv), dtype=np.uint64, count=n), out=koff[1:])
        np.cumsum(np.fromiter((len(v) for _, v in sorted_kv), dtype=np.uint64, count=n), out=voff[1:])
        keys = b"".join(k for k, _ in sorted_kv) + b"\0"
        vals = b"".join(v for _, v in sorted_kv) + b"\0"
        return self.lib.rsp_ingest_sorted(self.h, n, keys, koff.ctypes.data, vals, voff.ctypes.data,
                                          1 if allow_global_seqno else 0, None)

    def stats(self):
        st = Stats()
        self.lib.rsp_get_stats(self.h, C.byref(st))
        return {n: getattr(st, n) for n, _ in Stats._fields_}


class Engine:
    """One engine per GPU (shard_id -> GPU partitioning happens above, SURVEY §8e)."""

    def __init__(self, device=0, max_shards=0, arena_bytes=0, l0_compaction_trigger=0):
        self.lib = load_library()
        cfg = EngineCfg(abi_version=1, max_shards=max_shards, arena_bytes=arena_bytes,
                        l0_compaction_trigger=l0_compaction_trigger)
        h = C.c_void_p()
        rc = self.lib.rsp_engine_create(device, C.byref(cfg), C.byref(h))
        if rc != OK:
            raise RuntimeError(f"rsp_engine_create(device={device}) -> {rc}: no usable CUDA device "
                               "(the engine has no CPU fallback)")
        self.h = h
        self.device = device
        self.shards = {}

    def close(self):
        if self.h:
            for s in list(self.shards.values()):
                s.h = None
            self.lib.rsp_engine_destroy(self.h)
            self.h = None

    def open_shard(self, name, **kw):
        s = Shard(self, name, **kw)
        self.shards[name] = s
        return s

    # ---- batched calls (numpy in / numpy out; host memory) ----
    def apply_many(self, shard_ix, batches, ts_ms=None):
        """batches: list of bytes.  Returns int32 status per batch."""
        n = len(batches)
        six = np.ascontiguousarray(shard_ix, dtype=np.uint32)
        lens = np.fromiter((len(b) for b in batches), dtype=np.uint64, count=n)
        off = np.zeros(n + 1, dtype=np.uint64)
        np.cumsum(lens, out=off[1:])
        blob = np.frombuffer(b"".join(batches) + b"\0", dtype=np.uint8)
        return self.apply_packed(six, blob, off, ts_ms)

    def apply_packed(self, six, blob, off, ts_ms=None):
        n = len(six)
        st = np.zeros(n, dtype=np.int32)
        ts = None if ts_ms is None else np.ascontiguousarray(ts_ms, dtype=np.uint64)
        rc = self.lib.rsp_apply_many(self.h, n, _ptr(six), _ptr(blob), _ptr(off), _ptr(ts), _ptr(st))
        self.last_rc = rc  # (the call's own status: the first failing batch's, or an engine failure)
        return st

    def multi_get(self, shard_ix, keys, stride=256):
        """keys: list of bytes -> [(status, value|None)] with RocksDB MultiGet semantics."""
        n = len(keys)
        six = np.ascontiguousarray(shard_ix, dtype=np.uint32)
        off = np.zeros(n + 1, dtype=np.uint64)
        np.cumsum(np.fromiter((len(k) for k in keys), dtype=np.uint64, count=n), out=off[1:])
        blob = np.frombuffer(b"".join(keys) + b"\0", dtype=np.uint8)
        while True:
            vals = np.zeros(max(n * stride, 1), dtype=np.uint8)
            vlen = np.zeros(max(n, 1), dtype=np.uint32)
            st = np.zeros(max(n, 1), dtype=np.int32)
            rc = self.lib.rsp_multi_get(self.h, n, _ptr(six), _ptr(blob), _ptr(off), _ptr(vals), stride,
                                        _ptr(vlen), _ptr(st))
            if rc != OK:
                raise RuntimeError(f"rsp_multi_get -> {rc}")
            if n and (st[:n] == INCOMPLETE).any():
                stride = int(vlen[:n][st[:n] == INCOMPLETE].max())
                continue
            out = []
            for i in range(n):
                out.append((int(st[i]), vals[i * stride:i * stride + vlen[i]].tobytes() if st[i] == OK else None))
            return out

    def multi_get_fixed(self, six, keys, klen, vals, stride, vlen, st):
        """numpy arrays in place (pinned or pageable host memory)."""
        return self.lib.rsp_multi_get_fixed(self.h, len(six), _ptr(six), _ptr(keys), klen, _ptr(vals), stride,
                                            _ptr(vlen), _ptr(st))

    def multi_scan(self, shard_ix, keys, max_entries, stride):
        n = len(keys)
        six = np.ascontiguousarray(shard_ix, dtype=np.uint32)
        off = np.zeros(n + 1, dtype=np.uint64)
        np.cumsum(np.fromiter((len(k) for k in keys), dtype=np.uint64, count=n), out=off[1:])
        blob = np.frombuffer(b"".join(keys) + b"\0", dtype=np.uint8)
        out = np.zeros(max(n * stride, 1), dtype=np.uint8)
        n_out = np.zeros(max(n, 1), dtype=np.uint32)
        st = np.zeros(max(n, 1), dtype=np.int32)
        rc = self.lib.rsp_multi_scan(self.h, n, _ptr(six), _ptr(blob), _ptr(off), max_entries, _ptr(out), stride,
                                     _ptr(n_out), _ptr(st))
        if rc != OK:
            raise RuntimeError(f"rsp_multi_scan -> {rc}")
        res = []
        for i in range(n):
            recs, at = [], i * stride
            for _ in range(int(n_out[i])):
                kl = int(out[at:at + 4].view(np.uint32)[0])
                vl = int(out[at + 4:at + 8].view(np.uint32)[0])
                recs.append((out[at + 8:at + 8 + kl].tobytes(), out[at + 8 + kl:at + 8 + kl + vl].tobytes()))
                at += 8 + kl + vl
            res.append((int(st[i]), recs))
        return res

    def flush_all(self): return self.lib.rsp_flush_all(self.h)
    def compact_all(self): return self.lib.rsp_compact_all(self.h)
    def last_kernel_ms(self, what): return self.lib.rsp_last_kernel_ms(self.h, what.encode())
    def kernel_launches(self): return self.lib.rsp_kernel_launches(self.h)


class Router:
    """Several engines (one per GPU) behind one handle: shard_id -> engine fan-out of cross-shard batches
    (examples/counter_service/counter_router.cpp:36-66 inside one box)."""

    def __init__(self, engines):
        self.lib = load_library()
        self.engines = list(engines)
        arr = (C.c_void_p * len(self.engines))(*[e.h for e in self.engines])
        h = C.c_void_p()
        rc = self.lib.rsp_router_create(len(self.engines), arr, C.byref(h))
        if rc != OK:
            raise RuntimeError(f"rsp_router_create -> {rc}")
        self.h = h

    def close(self):
        if self.h:
            self.lib.rsp_router_destroy(self.h)
            self.h = None

    def add_shard(self, shard_id, shard):
        rc = self.lib.rsp_router_add_shard(self.h, shard_id, shard.h)
        if rc != OK:
            raise RuntimeError(f"rsp_router_add_shard({shard_id}) -> {rc}")

    def apply_many(self, shard_ids, batches, ts_ms=None):
        n = len(batches)
        ids = np.ascontiguousarray(shard_ids, dtype=np.uint32)
        off = np.zeros(n + 1, dtype=np.uint64)
        np.cumsum(np.fromiter((len(b) for b in batches), dtype=np.uint64, count=n), out=off[1:])
        blob = np.frombuffer(b"".join(batches) + b"\0", dtype=np.uint8)
        st = np.zeros(max(n, 1), dtype=np.int32)
        ts = None if ts_ms is None else np.ascontiguousarray(ts_ms, dtype=np.uint64)
        self.lib.rsp_router_apply_many(self.h, n, _ptr(ids), _ptr(blob), _ptr(off), _ptr(ts), _ptr(st))
        return st[:n]

    def multi_get(self, shard_ids, keys, stride=256):
        n = len(keys)
        ids = np.ascontiguousarray(shard_ids, dtype=np.uint32)
        off = np.zeros(n + 1, dtype=np.uint64)
        np.cumsum(np.fromiter((len(k) for k in keys), dtype=np.uint64, count=n), out=off[1:])
        blob = np.frombuffer(b"".join(keys) + b"\0", dtype=np.uint8)
        while True:
            vals = np.zeros(max(n * stride, 1), dtype=np.uint8)
            vlen = np.zeros(max(n, 1), dtype=np.uint32)
            st = np.zeros(max(n, 1), dtype=np.int32)
            rc = self.lib.rsp_router_multi_get(self.h, n, _ptr(ids), _ptr(blob), _ptr(off), _ptr(vals), stride, _ptr(vlen), _ptr(st))
            if n and (st[:n] == INCOMPLETE).any():
                stride = int(vlen[:n][st[:n] == INCOMPLETE].max())
                continue
            return [(int(st[i]), vals[i * stride:i * stride + vlen[i]].tobytes() if st[i] == OK else None) for i in range(n)], rc

    def multi_get_fixed(self, shard_ids, keys, klen, vals, stride, vlen, st):
        return self.lib.rsp_router_multi_get_fixed(self.h, len(shard_ids), _ptr(shard_ids), _ptr(keys), klen, _ptr(vals), stride,
                                                   _ptr(vlen), _ptr(st))
