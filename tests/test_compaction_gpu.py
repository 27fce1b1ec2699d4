"""Flush and compaction (csrc/k_compact.cu) checked run by run, entry by entry.

Reads cannot see everything a flush or a compaction gets wrong: a tombstone kept at the bottom, two heads for one key,
a hash slot off its probe sequence, a block-index entry one block off or a "uniform, all fixed Puts" flag on a run that
is not are all invisible to most lookups.  So after every flush, compaction and ingest in this file

  * every run of the shard is read back through rsp_debug_run and checked by `validate_run` (layout, order, padding,
    block index, hash index, descriptors on the host and on the device), and
  * the run the operation produced is compared byte for byte with `model_output`, a host model of the merge rules
    computed from the runs that took part (dumped before the operation) and the memtable (the test's own log of the
    operations applied since the shard's last flush), and
  * every key is read through get, multi_get, multi_get_fixed (16-byte keys) and a full scan and compared with the
    oracle port (oracle/okv.py), the semantic reference.

Merges run on the apply path (RSP_BG_COMPACT=0) so that which runs merge is deterministic, except in the one test
that leaves background merges on and checks every run with the validator and the oracle only.
"""
import ctypes as C
import os
import random
import struct
import time

import numpy as np
import pytest

from oracle import okv
from rocksplicator_b200.write_batch import WriteBatch

pytestmark = pytest.mark.gpu

EMUL = bool(os.environ.get("RSP_TEST_EMUL_LIB"))
T_DEL, T_PUT, T_MERGE, T_SDEL = 0, 1, 2, 7
NONE, COUNTER, UINT64ADD, APPEND = okv.MERGE_NONE, okv.MERGE_COUNTER, okv.MERGE_UINT64ADD, okv.MERGE_APPEND
OK, NOT_FOUND, BUSY = 0, 1, 11
RUN_ALL_PUT_FIXED = 1
FS_MAX_ITEMS = 24576   # k_flush_sort's shared-memory limit: larger memtables take the comparison sort
MERGE_TILE = 2048      # items per tile of the merge path
M64 = (1 << 64) - 1


# ---- the diagnostic read-back (include/rsp_b200.h: rsp_debug_run) ---------------------------------------------------
class RunDesc(C.Structure):
    _fields_ = [("heap", C.c_uint64), ("ent_off", C.c_uint64), ("hslots", C.c_uint64), ("blk_pfx", C.c_uint64)] + \
               [(n, C.c_uint32) for n in ("n_ent", "n_buckets", "ord_bits", "uniform_units", "n_blocks", "heap_units",
                                          "flags", "kv_len")]


class FastDesc(C.Structure):
    _fields_ = [("run0_heap", C.c_uint64), ("run0_hslots", C.c_uint64), ("n_buckets", C.c_uint32),
                ("meta", C.c_uint32), ("mt_count", C.c_uint32), ("merge_op", C.c_uint32)]


class RunInfo(C.Structure):
    _fields_ = [("n_runs", C.c_uint32), ("dev_n_runs", C.c_uint32), ("host", RunDesc), ("dev", RunDesc),
                ("fast_run", FastDesc), ("fast", FastDesc)]


def _desc(d):
    return {n: getattr(d, n) for n, _ in d._fields_}


class Run:
    """One run as dumped: descriptors, arrays and the decoded entries [(type, key, value, seq)]"""

    def __init__(self, info, heap, ent_off, blk_pfx, hslots):
        self.info = info
        self.host, self.dev = _desc(info.host), _desc(info.dev)
        self.fast_run, self.fast = _desc(info.fast_run), _desc(info.fast)
        self.id = info.host.heap
        self.heap, self.ent_off, self.blk_pfx, self.hslots = heap, ent_off, blk_pfx, hslots
        self.entries = []
        hb = heap.tobytes()
        self.hb = hb
        pos = 0
        for i in range(info.host.n_ent):
            st, kl, vl = struct.unpack_from("<QII", hb, pos * 16)
            k0 = pos * 16 + 16
            v0 = k0 + 16 * units(kl)
            self.entries.append((st & 0xff, hb[k0:k0 + kl], hb[v0:v0 + vl], st >> 8))
            pos += 1 + units(kl) + units(vl)


def dump_run(shard, r):
    """run r of the shard (0 = newest), or None.  Retries when a background merge replaced the run between the size
    query and the copy."""
    lib = shard.lib
    for _ in range(100):
        info = RunInfo()
        rc = lib.rsp_debug_run(shard.h, r, C.byref(info), None, None, None, None)
        if rc == NOT_FOUND:
            return None
        assert rc == OK, rc
        h = info.host
        heap = np.zeros(h.heap_units * 16, np.uint8)
        ent_off = np.zeros(h.n_ent, np.uint32)
        blk = np.zeros(h.n_blocks, np.uint64)
        hs = np.zeros(h.n_buckets * 8, np.uint32)
        rc = lib.rsp_debug_run(shard.h, r, C.byref(info), heap.ctypes.data, ent_off.ctypes.data, blk.ctypes.data,
                               hs.ctypes.data)
        if rc == NOT_FOUND:
            return None
        if rc == OK:
            return Run(info, heap, ent_off, blk, hs)
        assert rc == BUSY, rc
    raise AssertionError("the run kept changing")


def dump_all(shard):
    out = []
    while True:
        r = dump_run(shard, len(out))
        if r is None:
            return out
        out.append(r)


# ---- the run validator ----------------------------------------------------------------------------------------------
def units(n):
    return (n + 15) >> 4


def hash_key(key):
    """hash_key_padded of format.cuh"""
    n = len(key)
    h = (0x5EED0001D1B54A32 ^ (n * 0x9E3779B97F4A7C15)) & M64
    padded = key + bytes(-n % 8)
    for i in range(0, len(padded), 8):
        w = int.from_bytes(padded[i:i + 8], "little")
        h = ((h ^ w) * 0xff51afd7ed558ccd) & M64
        h ^= h >> 32
    h ^= h >> 33
    h = (h * 0xc4ceb9fe1a85ec53) & M64
    h ^= h >> 29
    return h


def prefix_be(key):
    return int.from_bytes((key + bytes(8))[:8], "big")


def validate_run(run):
    """every structural invariant of one run (see the module docstring); returns the number of distinct keys"""
    h, hb, ents = run.host, run.hb, run.entries
    n = h["n_ent"]
    assert n > 0 and len(ents) == n
    # restart array, entry layout, padding
    pos = 0
    assert run.ent_off[0] == 0
    for i in range(n):
        assert run.ent_off[i] == pos, ("ent_off", i, int(run.ent_off[i]), pos)
        _, kl, vl = struct.unpack_from("<QII", hb, pos * 16)
        k0 = pos * 16 + 16
        v0 = k0 + 16 * units(kl)
        end = v0 + 16 * units(vl)
        assert hb[k0 + kl:v0] == bytes(v0 - k0 - kl), ("key padding", i)
        assert hb[v0 + vl:end] == bytes(end - v0 - vl), ("value padding", i)
        pos += 1 + units(kl) + units(vl)
    assert pos == h["heap_units"], ("heap_units", pos, h["heap_units"])
    # order: keys ascending (bytewise, shorter first), versions of one key newest first; the first version of each key
    heads = []
    for i, (t, k, v, seq) in enumerate(ents):
        assert t in (T_DEL, T_PUT, T_MERGE, T_SDEL), ("type", i, t)
        if i == 0 or ents[i - 1][1] != k:
            assert i == 0 or ents[i - 1][1] < k, ("key order", i, ents[i - 1][1], k)
            heads.append(i)
        else:
            assert ents[i - 1][3] > seq, ("version order", i, k, ents[i - 1][3], seq)
    # block index
    assert h["n_blocks"] == (n + 31) // 32
    for b in range(h["n_blocks"]):
        assert int(run.blk_pfx[b]) == prefix_be(ents[32 * b][1]), ("blk_pfx", b)
    # hash index: sized for the distinct keys; every key's head found by probing from its home bucket
    keys = len(heads)
    assert h["n_buckets"] == max(1, (keys + 3) // 4), ("n_buckets", h["n_buckets"], keys)
    assert h["ord_bits"] == n.bit_length(), ("ord_bits", h["ord_bits"], n)
    ob, nb = h["ord_bits"], h["n_buckets"]
    slots = run.hslots.reshape(nb, 8)
    head_set = set(heads)
    nz = slots[slots != 0]
    assert len(nz) == keys, ("hash slots", len(nz), keys)
    for val in nz.tolist():
        assert (val & ((1 << ob) - 1)) - 1 in head_set, ("slot points at a non-head", val)
    for i in heads:
        hh = hash_key(ents[i][1])
        want = ((((hh >> 32) >> ob) << ob) | (i + 1)) & 0xffffffff
        b = ((hh & 0xffffffff) * nb) >> 32
        for _ in range(nb):
            row = slots[b]
            if want in row:
                break
            assert 0 not in row, ("probe ends before the key's slot", i, ents[i][1])
            b = 0 if b + 1 == nb else b + 1
        else:
            raise AssertionError(("key not in its probe sequence", i))
    # uniform size, all-fixed-Put flag
    sizes = {1 + units(len(k)) + units(len(v)) for _, k, v, _ in ents}
    assert h["uniform_units"] == (sizes.pop() if len(sizes) == 1 else 0), ("uniform_units", h["uniform_units"])
    shapes = {(t, len(k), len(v)) for t, k, v, _ in ents}
    fixed = len(shapes) == 1 and next(iter(shapes))[0] == T_PUT
    if fixed:
        _, kl, vl = next(iter(shapes))
        fixed = kl <= 0xffff and vl <= 0xffff  # (kv_len packs both in 16 bits)
    assert bool(h["flags"] & RUN_ALL_PUT_FIXED) == fixed, ("RUN_ALL_PUT_FIXED", h["flags"], shapes if len(shapes) < 4 else len(shapes))
    assert h["kv_len"] == ((kl | vl << 16) if fixed else 0), ("kv_len", h["kv_len"])
    # what the readers use: ShardDev.runs[r], the per-run fast descriptor and (run 0) the shard's fast descriptor
    assert run.dev == h, ("device descriptor", run.dev, h)
    assert run.info.dev_n_runs == run.info.n_runs
    meta = ob | min(h["uniform_units"], 255) << 8
    assert run.fast_run == {"run0_heap": h["heap"], "run0_hslots": h["hslots"], "n_buckets": nb, "meta": meta,
                            "mt_count": 0, "merge_op": 0}, ("fast_runs row", run.fast_run)
    return keys


def validate_shard(shard, runs=None, merge_op=None):
    """validate_run on every run of the shard; the shard's fast descriptor from run 0"""
    runs = dump_all(shard) if runs is None else runs
    for i, r in enumerate(runs):
        validate_run(r)
        if i == 0:
            f = r.fast
            h = r.host
            meta = h["ord_bits"] | min(h["uniform_units"], 255) << 8 | min(r.info.n_runs, 255) << 16 | 1 << 24
            assert (f["run0_heap"], f["run0_hslots"], f["n_buckets"], f["meta"]) == (h["heap"], h["hslots"], h["n_buckets"], meta), \
                ("ShardFast", f, h)
            assert merge_op is None or f["merge_op"] == merge_op
    return runs


# ---- the model of a flush / compaction ------------------------------------------------------------------------------
def u64(b):
    return int.from_bytes(b, "little")


def fold_group(g, merge_op, bottom):
    """the versions of one key, newest first -> what the output keeps (k_compact_size's keep and fold rules)"""
    t0 = g[0][0]
    if t0 == T_PUT:
        return [g[0]]
    if t0 != T_MERGE:
        return [] if bottom else [g[0]]
    m = 0
    while m < len(g) and g[m][0] == T_MERGE:
        m += 1
    ops, base = g[:m], (g[m] if m < len(g) else None)
    bad = sum(1 for e in ops if len(e[2]) != 8)
    s = sum(u64(e[2]) for e in ops if len(e[2]) == 8) & M64
    _, key, _, seq = g[0]
    imm = lambda t, v: [(t, key, struct.pack("<Q", v & M64), seq)]  # noqa: E731
    if merge_op in (COUNTER, UINT64ADD):
        if base is not None and base[0] == T_PUT:
            bv = base[2]
            if merge_op == COUNTER:
                if bad == 0 and len(bv) == 8:
                    return imm(T_PUT, s + u64(bv))
            else:
                return imm(T_PUT, s + (u64(bv) if len(bv) == 8 else 0))
        elif base is not None or bottom:
            if merge_op == COUNTER:
                if len(ops) == 1:
                    return [(T_PUT, key, ops[0][2], seq)]
                if bad == 0:
                    return imm(T_PUT, s)
            else:
                return imm(T_PUT, s)
        elif len(ops) >= 2 and (merge_op == UINT64ADD or bad == 0):
            return imm(T_MERGE, s)
    keep = list(ops)
    if base is not None and (base[0] == T_PUT or not bottom):
        keep.append(base)
    return keep


def model_output(sources, merge_op, bottom):
    """sources: lists of (type, key, value, seq), newest source first, each in its stored order (the memtable newest
    first) -> the output run's entries"""
    items = [(e[1], si, p, e) for si, src in enumerate(sources) for p, e in enumerate(src)]
    items.sort(key=lambda x: x[:3])
    out, i = [], 0
    while i < len(items):
        j = i
        while j < len(items) and items[j][0] == items[i][0]:
            j += 1
        out += fold_group([x[3] for x in items[i:j]], merge_op, bottom)
        i = j
    return out


def serialize(entries):
    """run heap bytes and ent_off of entries [(type, key, value, seq)]"""
    parts, offs, pos = [], [], 0
    for t, k, v, seq in entries:
        offs.append(pos)
        e = struct.pack("<QII", (seq << 8) | t, len(k), len(v)) + k + bytes(-len(k) % 16) + v + bytes(-len(v) % 16)
        parts.append(e)
        pos += len(e) // 16
    return b"".join(parts), offs


def expect_comparison_sort(mem):
    """does k_flush_sort hand this memtable (newest first) to the comparison sort?"""
    if len(mem) < 2:
        return False
    if len(mem) > FS_MAX_ITEMS:
        return True
    pf = [prefix_be(e[1]) for e in mem]
    if (min(pf) ^ max(pf)).bit_length() > 48:
        return True
    by = {}
    for e in mem:
        by.setdefault(prefix_be(e[1]), set()).add(e[1])
    return any(len(v) > 1 for v in by.values())


# ---- shards and their oracles ---------------------------------------------------------------------------------------
_port = [None]


def port():
    if _port[0] is None:
        _port[0] = okv.load_port()
    return _port[0]


def batch_of(ops):
    wb = WriteBatch()
    for t, k, v in ops:
        if t == T_PUT:
            wb.put(k, v)
        elif t == T_MERGE:
            wb.merge(k, v)
        elif t == T_DEL:
            wb.delete(k)
        else:
            wb.single_delete(k)
    return wb.data()


class Twin:
    """one engine shard, its oracle, the log of what its memtable holds and the shape of the last operation"""
    _n = [0]

    def __init__(self, eng, merge_op=NONE, wb=1 << 20):
        Twin._n[0] += 1
        self.eng = eng
        self.merge_op = merge_op
        self.s = eng.open_shard("c%05d" % Twin._n[0], merge_op=merge_op, write_buffer_bytes=wb)
        self.o = okv.Okv(port(), merge_op=merge_op)
        self.log = []        # the memtable: (type, key, value, seq) in apply order since the last flush
        self.keys = set()
        self.seq_delta = 0   # engine sequence - oracle sequence (an ingest moves them apart)
        self.flushes = 0

    def write(self, ops, chunk=4096):
        """ops: [(type, key, value)]; applied as WriteBatches of up to `chunk` operations"""
        for c0 in range(0, len(ops), chunk):
            part = ops[c0:c0 + chunk]
            d = batch_of(part)
            seq0 = self.o.latest_seq() + self.seq_delta
            rc, ro = self.s.apply(d, 7), self.o.apply(d, 7)
            assert rc == ro, (rc, ro, self.s.last_error, self.o.last_error)
            if rc == OK:
                self.log += [(t, k, v, seq0 + 1 + i) for i, (t, k, v) in enumerate(part)]
                self.keys.update(k for _, k, _ in part)
            assert self.s.latest_seq() == self.o.latest_seq() + self.seq_delta
        assert self.s.stats()["flushes"] == self.flushes, "a flush nobody asked for (write buffer too small)"

    def ingest(self, kv):
        """rsp_ingest_sorted of sorted (key, value) pairs; the oracle applies them as Puts"""
        before = self.s.latest_seq()
        runs0 = dump_all(self.s)
        overlap = any(r.entries[0][1] <= kv[-1][0] and kv[0][0] <= r.entries[-1][1] for r in runs0)
        assert self.s.ingest(kv) == OK, self.s.last_error
        d = WriteBatch()
        for k, v in kv:
            d.put(k, v)
        assert self.o.apply(d.data(), 7) == OK
        self.keys.update(k for k, _ in kv)
        self.seq_delta += (1 if overlap else 0) - len(kv)
        assert self.s.latest_seq() == before + (1 if overlap else 0)
        runs = validate_shard(self.s, merge_op=self.merge_op)
        assert [r.id for r in runs[1:]] == [r.id for r in runs0] and runs[0].id not in {r.id for r in runs0}
        assert [(k, v) for _, k, v, _ in runs[0].entries] == list(kv)
        assert all(t == T_PUT and seq == self.s.latest_seq() for t, _, _, seq in runs[0].entries)

    def close(self):
        self.s.close()
        self.o.close()


def check_reads(t, n_get=48):
    """every key through multi_get (and multi_get_fixed for 16-byte keys), a sample through get, a full scan"""
    keys = sorted(t.keys)
    probe = keys + [b"\xff" * 17, b"zz-missing"]
    assert t.s.multi_get(probe) == t.o.multi_get(probe), "multi_get"
    rng = random.Random(len(keys))
    for k in rng.sample(probe, min(n_get, len(probe))):
        assert t.s.get(k) == t.o.get(k), ("get", k)
    k16 = [k for k in keys if len(k) == 16]
    if k16:
        q = k16 + [bytes(15) + b"\x01"]
        n, stride = len(q), 4096
        vals = np.zeros((n, stride), np.uint8)
        vlen = np.zeros(n, np.uint32)
        st = np.zeros(n, np.int32)
        assert t.eng.multi_get_fixed(np.full(n, t.s.index, np.uint32), np.frombuffer(b"".join(q), np.uint8).copy(), 16,
                                     vals, stride, vlen, st) == OK
        for i, (w_st, w_v) in enumerate(t.o.multi_get(q)):
            if w_st == OK and len(w_v) > stride:
                assert st[i] == 7
                continue
            assert st[i] == w_st, ("multi_get_fixed", i, int(st[i]), w_st)
            if w_st == OK:
                assert bytes(vals[i, :vlen[i]]) == w_v, ("multi_get_fixed value", i)
    assert t.s.scan() == t.o.scan(), "scan"


class Op:
    """before / after one flush or compaction of a twin: the transition is checked against the model"""

    def __init__(self, t):
        self.t = t
        self.before = dump_all(t.s)
        self.mem = list(reversed(t.log))
        self.stats = t.s.stats()

    def check(self, want_merged=None):
        t = self.t
        after = validate_shard(t.s, merge_op=t.merge_op)
        st = t.s.stats()
        b_ids, a_ids = [r.id for r in self.before], [r.id for r in after]
        new = [i for i in a_ids if i not in b_ids]
        assert len(new) <= 1, "more than one new run"
        gone = [i for i, r in enumerate(b_ids) if r not in a_ids]
        assert gone == list(range(gone[0], gone[0] + len(gone))) if gone else True, "merged runs not contiguous"
        at = gone[0] if gone else 0
        if new:
            assert a_ids.index(new[0]) == at
        assert [i for i in a_ids if i != (new[0] if new else None)] == b_ids[:at] + b_ids[at + len(gone):], "run order"
        bottom = at + len(gone) == len(b_ids)
        if want_merged is not None:
            assert len(gone) == want_merged, ("runs merged", len(gone), want_merged)
        sources = ([self.mem] if self.mem else []) + [self.before[i].entries for i in gone]
        want = model_output(sources, t.merge_op, bottom) if sources else []
        if new:
            got = after[a_ids.index(new[0])]
            heap, offs = serialize(want)
            if got.hb != heap:
                first = next(i for i in range(min(len(want), len(got.entries)) + 1)
                             if i == len(want) or i == len(got.entries) or want[i] != got.entries[i])
                raise AssertionError(("output differs from the model", "bottom", bottom, "entry", first,
                                      want[first:first + 3], got.entries[first:first + 3], len(want), len(got.entries)))
            assert got.ent_off.tolist() == offs
        else:
            assert not want, ("no output run, the model keeps", len(want))
        # counters
        assert st["memtable_entries"] == 0 and st["flushes"] == self.stats["flushes"] + (1 if self.mem else 0)
        assert st["compactions"] == self.stats["compactions"] + (1 if gone else 0)
        assert st["flush_comparison_sorts"] == self.stats["flush_comparison_sorts"] + \
            (1 if self.mem and expect_comparison_sort(self.mem) else 0), "flush_comparison_sorts"
        assert st["n_runs"] == len(after)
        assert st["run_entries"] == sum(r.host["n_ent"] for r in after)
        assert st["run_bytes"] == sum(r.host["heap_units"] * 16 for r in after)
        t.flushes = st["flushes"]
        t.log.clear()
        return bottom, len(gone)


def flush(t, check_reads_too=True, **kw):
    op = Op(t)
    assert t.s.flush() == OK
    res = op.check(**kw)
    if check_reads_too:
        check_reads(t)
    return res


def compact(t, check_reads_too=True, **kw):
    op = Op(t)
    assert t.s.compact() == OK
    res = op.check(**kw)
    assert res[0], "a full compaction is a bottom output"
    if check_reads_too:
        check_reads(t)
    return res


# ---- engines --------------------------------------------------------------------------------------------------------
@pytest.fixture
def engine_factory():
    """engine_factory(trigger, bg=False): one engine at a time; merges on the apply path unless bg"""
    from rocksplicator_b200 import engine
    state = {"eng": None, "twins": []}
    old = os.environ.get("RSP_BG_COMPACT")

    def make(trigger, bg=False, max_shards=64):
        close()
        if bg:
            os.environ.pop("RSP_BG_COMPACT", None)
        else:
            os.environ["RSP_BG_COMPACT"] = "0"  # read in rsp_engine_create
        state["eng"] = engine.Engine(0, max_shards=max_shards, l0_compaction_trigger=trigger)
        return state["eng"]

    def close():
        for t in state["twins"]:
            t.o.close()
        state["twins"].clear()
        if state["eng"] is not None:
            state["eng"].close()
            state["eng"] = None

    make.twin = lambda *a, **kw: state["twins"].append(Twin(state["eng"], *a, **kw)) or state["twins"][-1]
    yield make
    close()
    if old is None:
        os.environ.pop("RSP_BG_COMPACT", None)
    else:
        os.environ["RSP_BG_COMPACT"] = old


def wb_for(n_ops, payload=0):
    """a write buffer that holds n_ops entries and `payload` key + value bytes without flushing"""
    return (1 << 20) + 16 * 7 * 3 * n_ops + 3 * payload


# ---- workloads ------------------------------------------------------------------------------------------------------
def k16(rng, n, prefix=b""):
    out = set()
    while len(out) < n:
        out.add(prefix + rng.randbytes(16 - len(prefix)))
    return sorted(out)


def operand(rng, merge_op, bad_frac=0.1):
    if merge_op in (COUNTER, UINT64ADD):
        return rng.randbytes(rng.choice([3, 9])) if rng.random() < bad_frac else struct.pack("<q", rng.randint(-99, 99))
    return rng.randbytes(rng.choice([1, 8, 20]))


def mixed_ops(rng, keys, n, merge_op=COUNTER, p_del=0.12, p_sdel=0.04, p_merge=0.25, vlens=(8, 8, 16, 64, 100)):
    ops = []
    for _ in range(n):
        k = rng.choice(keys)
        r = rng.random()
        if r < p_del:
            ops.append((T_DEL, k, b""))
        elif r < p_del + p_sdel:
            ops.append((T_SDEL, k, b""))
        elif r < p_del + p_sdel + p_merge:
            ops.append((T_MERGE, k, operand(rng, merge_op)))
        else:
            ops.append((T_PUT, k, rng.randbytes(rng.choice(vlens))))
    return ops


def puts(rng, keys, vlen=24):
    return [(T_PUT, k, rng.randbytes(vlen)) for k in keys]


def keys_with_spread(rng, n, v, suffix=8):
    """n distinct 8-byte prefixes whose min ^ max has bit length v (+ a random suffix)"""
    base = 0x5A5A5A5A5A5A5A5A & ~((1 << v) - 1) if v < 64 else 0
    if v == 0:
        return [base.to_bytes(8, "big") + rng.randbytes(suffix)]
    pf = {base, base | (1 << (v - 1))}
    while len(pf) < min(n, 1 << v):
        pf.add(base | rng.getrandbits(v))
    return sorted(p.to_bytes(8, "big") + rng.randbytes(suffix) for p in pf)


# ---- k_flush_sort: the radix sort of a memtable ---------------------------------------------------------------------
@pytest.mark.parametrize("trigger", [4, 8])
def test_radix_flush_counts(engine_factory, trigger):
    """memtables of 2 .. 4097 entries flushed onto a growing run stack: tiered merges at trigger 4, deep stacks at 8"""
    rng = random.Random(trigger)
    engine_factory(trigger)
    t = engine_factory.twin(COUNTER, wb=wb_for(5000, 5000 * 100))
    pool = k16(rng, 3000, prefix=b"\x01\x02")  # V <= 48: the radix path
    for n in (2, 31, 32, 33, 511, 512, 513, 4097):
        t.write(mixed_ops(rng, pool, n))
        assert not expect_comparison_sort(list(reversed(t.log)))
        flush(t)
    compact(t)


@pytest.mark.parametrize("n", [FS_MAX_ITEMS - 1, FS_MAX_ITEMS, FS_MAX_ITEMS + 1])
def test_flush_sort_item_limit(engine_factory, n):
    """24,575 and 24,576 entries fit the radix sort's shared memory, 24,577 take the comparison sort"""
    rng = random.Random(n)
    engine_factory(8)
    t = engine_factory.twin(UINT64ADD, wb=wb_for(n, n * 40))
    pool = keys_with_spread(rng, n // 2, 40)
    t.write(puts(rng, pool[:200]))
    flush(t)
    t.write(mixed_ops(rng, pool, n, UINT64ADD, vlens=(8, 16)))
    assert expect_comparison_sort(list(reversed(t.log))) == (n > FS_MAX_ITEMS)
    flush(t, want_merged=0)
    compact(t)


@pytest.mark.parametrize("v", [0, 8, 9, 16, 17, 48, 49])
def test_flush_sort_prefix_spread(engine_factory, v):
    """prefix spreads V: no pass (0), an even / odd number of passes (8 / 9, 16 / 17), the last one that fits beside
    the rank (48) and the first that does not (49)"""
    rng = random.Random(v)
    engine_factory(4)
    t = engine_factory.twin(COUNTER, wb=wb_for(3000, 3000 * 70))
    pool = keys_with_spread(rng, 600, v)
    t.write(mixed_ops(rng, pool, 1500 if v else 1200))
    if v == 0:  # all versions of one key: more than one thread's chunk, more than 1,024 versions
        assert len({e[1] for e in t.log}) == 1
    mem = list(reversed(t.log))
    pf = [prefix_be(e[1]) for e in mem]
    assert (min(pf) ^ max(pf)).bit_length() == v
    assert expect_comparison_sort(mem) == (v > 48)
    flush(t)
    t.write(mixed_ops(rng, pool, 700))
    flush(t)
    compact(t)


def test_short_keys_and_zero_padding(engine_factory):
    """keys shorter than 8 bytes next to the same bytes with zeros appended, and the empty key: distinct keys with one
    padded prefix (the comparison sort), and short keys with distinct prefixes (the radix sort)"""
    rng = random.Random(5)
    engine_factory(4)
    t = engine_factory.twin(COUNTER)
    tricky = [b"", b"\0", b"\0\0", b"\0" * 8, b"\0" * 9, b"a", b"a\0", b"a\0\0\0", b"a\0" * 4, b"a" + bytes(8), b"ab",
              b"ab\0", b"\x01", b"\xff", b"\xff\0", b"\xff" * 8, b"\xff" * 9]
    t.write(mixed_ops(rng, tricky, 400))
    assert expect_comparison_sort(list(reversed(t.log)))
    flush(t)
    distinct = [b"BB"] + [b"BB" + bytes([i]) for i in range(1, 256)] + [b"BB" + bytes([i, 7]) for i in range(0, 256, 3)]
    t.write(mixed_ops(rng, distinct, 500))
    assert not expect_comparison_sort(list(reversed(t.log)))
    flush(t)
    t.write(mixed_ops(rng, tricky + distinct, 300))
    flush(t)
    compact(t)


# ---- k_compact_sort: the bitonic sort ------------------------------------------------------------------------------
BITONIC_SIZES = [4096, 4097, 8193, 16385, 40000]


@pytest.mark.parametrize("n", BITONIC_SIZES)
def test_bitonic_sort_sizes(engine_factory, n):
    """shared-prefix memtables: one tile (4,096), just past it, and several global-memory stages (40,000 -> 65,536);
    about three versions per key, so newest-first within a key rests on the tie-break"""
    rng = random.Random(n)
    engine_factory(8)
    t = engine_factory.twin(COUNTER, wb=wb_for(n, n * 40))
    pool = k16(rng, max(2, n // 3), prefix=b"SHAREDPF")
    t.write(puts(rng, pool[: len(pool) // 2], 8))
    flush(t, check_reads_too=False)
    t.write(mixed_ops(rng, pool, n, vlens=(8, 24)))
    assert expect_comparison_sort(list(reversed(t.log)))
    flush(t, want_merged=0)
    compact(t)


# ---- merge path -----------------------------------------------------------------------------------------------------
def build_stack(t, rng, sizes, pool, merge_op=COUNTER):
    """one flushed run per size (newest last) at trigger 8: no merges up to 7 runs"""
    for n in sizes:
        t.write(mixed_ops(rng, pool, n, merge_op))
        flush(t, check_reads_too=False, want_merged=0)


@pytest.mark.parametrize("n_src", [2, 3, 5, 8, 9])
def test_merge_sources(engine_factory, n_src):
    """2 to 9 sources merged in one compaction (9: 7 flushed runs, an ingested run and the memtable)"""
    rng = random.Random(n_src)
    engine_factory(8)
    t = engine_factory.twin(COUNTER, wb=wb_for(4000, 400000))
    pool = k16(rng, 1500, prefix=b"\x03")
    n_runs = n_src - 1
    build_stack(t, rng, [rng.randint(50, 900) for _ in range(min(n_runs, 7))], pool)
    if n_runs == 8:
        ing = sorted({rng.choice(pool) for _ in range(500)} | {b"\x03ingest%09d" % i for i in range(40)})
        t.ingest([(k, rng.randbytes(8)) for k in ing])
    t.write(mixed_ops(rng, pool, 1200))
    assert len(dump_all(t.s)) == n_runs
    compact(t, want_merged=n_runs)


@pytest.mark.parametrize("total", [2047, 2048, 2049, 2 * 2048 - 1, 2 * 2048 + 1, 5 * 2048 - 1, 5 * 2048 + 1])
def test_merge_tile_boundaries(engine_factory, total):
    """item totals at and around the 2,048-item merge tiles, over 2 and 3 sources"""
    rng = random.Random(total)
    engine_factory(8)
    t = engine_factory.twin(UINT64ADD, wb=wb_for(total, total * 40))
    pool = k16(rng, total, prefix=b"\x04\x04")
    a = total // 3
    t.write(puts(rng, rng.sample(pool, a), 8))
    flush(t, check_reads_too=False)
    if total % 2:
        b = total // 4
        t.write(puts(rng, rng.sample(pool, b), 8))
        flush(t, check_reads_too=False)
        a += b
    t.write(mixed_ops(rng, pool, total - a, UINT64ADD))
    op = Op(t)
    assert sum(r.host["n_ent"] for r in op.before) + len(t.log) == total
    assert t.s.compact() == OK
    op.check()
    check_reads(t)


@pytest.mark.parametrize("skew", ["run_big", "mem_big"])
def test_merge_skewed_sources(engine_factory, skew):
    """one entry beside 10,000"""
    rng = random.Random(len(skew))
    engine_factory(8)
    t = engine_factory.twin(COUNTER, wb=wb_for(10001, 10001 * 40))
    pool = k16(rng, 10000, prefix=b"\x05")
    big, small = puts(rng, pool, 8), [(T_PUT, rng.choice(pool), b"one")]
    t.write(big if skew == "run_big" else small)
    flush(t, check_reads_too=False)
    t.write(small if skew == "run_big" else big)
    compact(t, want_merged=1)
    t.write([(T_DEL, pool[0], b""), (T_PUT, pool[-1] + b"x", b"after")])
    compact(t, want_merged=1)


def test_hot_key_across_tiles(engine_factory):
    """one key with operand stacks in all 9 sources (2,700 versions: the merge tiles and the co-rank splits fall inside
    its group), beside distinct keys that share its 8-byte prefix in other runs"""
    rng = random.Random(9)
    engine_factory(8)
    t = engine_factory.twin(APPEND, wb=wb_for(6000, 6000 * 40))
    hot = b"HOTKEY__middle"
    near = [b"HOTKEY__" + rng.randbytes(rng.choice([1, 8, 12])) for _ in range(600)]
    others = k16(rng, 800)
    for r in range(7):
        ops = [(T_MERGE, hot, b"op%d.%d" % (r, i)) for i in range(300)]
        ops += mixed_ops(rng, near[r * 80:(r + 1) * 80] + others, 250, APPEND)
        rng.shuffle(ops)
        t.write(ops)
        flush(t, check_reads_too=(r == 6), want_merged=0)
    t.ingest(sorted([(hot, b"ingested")] + [(k, b"i") for k in set(near[560:590])]))
    t.write([(T_MERGE, hot, b"mem%d" % i) for i in range(300)] + mixed_ops(rng, near + others, 400, APPEND))
    versions = sum(1 for r in dump_all(t.s) for e in r.entries if e[1] == hot) + sum(1 for e in t.log if e[1] == hot)
    assert versions > MERGE_TILE
    compact(t, want_merged=8)


def test_ingest_under_operands(engine_factory):
    """Merge operands flushed onto ingested Puts of a young shard (sequence numbers below the ingested run's size):
    the ingested run carries the ingest's sequence number, so the kept stack and its base stay newest first"""
    rng = random.Random(16)
    engine_factory(8)
    t = engine_factory.twin(APPEND)
    keys = k16(rng, 300, prefix=b"\x08")
    t.write([(T_PUT, k, b"old") for k in keys[:5]])
    flush(t)
    t.ingest([(k, b"ingested") for k in keys])  # overlaps: the global seqno
    t.write([(T_MERGE, k, b"+%d" % i) for i, k in enumerate(keys[::2])])
    flush(t)
    t.ingest([(b"\x09" + k, b"far") for k in keys[:50]])  # no overlap: the current sequence number
    t.write([(T_MERGE, b"\x09" + k, b"+") for k in keys[:50:3]])
    compact(t, want_merged=4)


# ---- k_compact_size: keep and fold ---------------------------------------------------------------------------------
@pytest.mark.parametrize("merge_op", [NONE, COUNTER, UINT64ADD, APPEND])
@pytest.mark.parametrize("trigger", [4, 8])
def test_keep_and_fold(engine_factory, merge_op, trigger):
    """every merge operator with good and bad operands, Put / Delete / SingleDelete / no bases, at the bottom and not:
    a big bottom run, then small flushes onto it (a tiered merge of the small runs at trigger 4), then a full
    compaction"""
    rng = random.Random(merge_op * 10 + trigger)
    engine_factory(trigger)
    t = engine_factory.twin(merge_op, wb=wb_for(4000, 4000 * 40))
    pool = k16(rng, 400, prefix=b"\x06")
    t.write(puts(rng, pool, 8) + [(T_PUT, k, b"odd") for k in pool[::17]])
    flush(t)
    scripted = pool[:24]
    for stage in range(5):
        ops = mixed_ops(rng, pool[24:], 120, merge_op, p_del=0.15, p_sdel=0.1, p_merge=0.5)
        # scripted keys: one operand at the bottom, wrong-size operands, Delete / SingleDelete bases, long stacks
        for i, k in enumerate(scripted):
            kind = (i + stage) % 6
            if kind == 0:
                ops.append((T_MERGE, k, operand(rng, merge_op, 0)))
            elif kind == 1:
                ops.append((T_MERGE, k, b"bad"))
            elif kind == 2:
                ops += [(T_DEL, k, b""), (T_MERGE, k, operand(rng, merge_op, 0))]
            elif kind == 3:
                ops += [(T_SDEL, k, b""), (T_MERGE, k, operand(rng, merge_op, 0)), (T_MERGE, k, operand(rng, merge_op, 0))]
            elif kind == 4:
                ops += [(T_PUT, k, b"base-not-8"), (T_MERGE, k, operand(rng, merge_op, 0))]
            else:
                ops += [(T_MERGE, k, operand(rng, merge_op, 0.3)) for _ in range(3)]
        t.write(ops)
        flush(t)
    fresh = [b"\x07single%04d" % i for i in range(30)]  # a single operand, no base, at the bottom
    t.write([(T_MERGE, k, operand(rng, merge_op, 0.5)) for k in fresh] + [(T_SDEL, k, b"") for k in pool[100:140]])
    t.keys.update(fresh)
    compact(t)


def test_long_groups(engine_factory):
    """one key with 1,500 versions and a key with 1,100 operands: groups longer than one thread's chunk"""
    rng = random.Random(11)
    engine_factory(4)
    t = engine_factory.twin(UINT64ADD, wb=wb_for(5000, 5000 * 40))
    a, b = b"A" * 16, b"B" * 16
    t.write([(T_PUT, a, struct.pack("<Q", i)) for i in range(1500)] +
            [(T_MERGE, b, operand(rng, UINT64ADD, 0.2)) for _ in range(1100)] + puts(rng, k16(rng, 300), 8))
    flush(t)
    t.write([(T_MERGE, a, struct.pack("<Q", 1)) for _ in range(1200)] + [(T_DEL, b, b"")] +
            [(T_MERGE, b, struct.pack("<Q", 2)) for _ in range(1100)])
    flush(t)
    compact(t)


def test_huge_key_and_value(engine_factory):
    """klen / vlen above 0xFFFF (the uncached shape path of k_compact_size)"""
    rng = random.Random(12)
    engine_factory(4)
    t = engine_factory.twin(COUNTER, wb=wb_for(200, 400000))
    big_v, big_k = rng.randbytes(70000), b"K" * 70000
    t.write(puts(rng, k16(rng, 50), 8) + [(T_PUT, b"bigvalue", big_v)])
    flush(t)
    t.write([(T_PUT, big_k, b"v"), (T_MERGE, b"bigvalue", struct.pack("<Q", 1))])
    assert t.s.get(big_k) == (OK, b"v")
    flush(t)
    compact(t)


# ---- descriptors ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("uni", [254, 255, 256])
def test_uniform_units_around_the_fast_field(engine_factory, uni):
    """runs whose entries are all `uni` units: ShardFast's U is 8 bits (255 = too large for the fast kernels)"""
    rng = random.Random(uni)
    engine_factory(4)
    t = engine_factory.twin(NONE, wb=wb_for(200, 200 * 5000))
    keys = k16(rng, 40)
    vlen = (uni - 2) * 16
    t.write(puts(rng, keys, vlen))
    flush(t)
    assert dump_all(t.s)[0].host["uniform_units"] == uni
    t.write(puts(rng, keys[::3], vlen - 5))  # same size in units, another vlen: uniform, not all fixed
    flush(t)
    compact(t)


def test_all_put_fixed_decision(engine_factory):
    """an all-fixed-Put run next to runs with one Delete, one odd-length value (same units), one shorter key"""
    rng = random.Random(13)
    engine_factory(8)
    t = engine_factory.twin(NONE)
    keys = k16(rng, 200)
    t.write(puts(rng, keys, 64))
    flush(t)
    assert dump_all(t.s)[0].host["flags"] & RUN_ALL_PUT_FIXED
    t.write(puts(rng, keys[:50], 64) + [(T_DEL, keys[60], b"")])
    flush(t)
    t.write(puts(rng, keys[:50], 64) + [(T_PUT, keys[70], rng.randbytes(63))])
    flush(t)
    r = dump_all(t.s)[0]
    assert r.host["uniform_units"] == 6 and not r.host["flags"] & RUN_ALL_PUT_FIXED
    t.write(puts(rng, keys[:50], 64) + [(T_PUT, keys[80][:15], rng.randbytes(64))])
    t.keys.add(keys[80][:15])
    flush(t)
    t.write(puts(rng, keys, 64) + [(T_DEL, keys[80][:15], b"")])
    compact(t)
    assert dump_all(t.s)[0].host["flags"] & RUN_ALL_PUT_FIXED


# ---- batches of shards ---------------------------------------------------------------------------------------------
def test_batched_flush_and_compact_all(engine_factory):
    """one rsp_flush_all and one rsp_compact_all over 40 shards of different shapes (one k_flush_sort cap and one merge
    grid shared by all): memtable only, runs only, above FS_MAX_ITEMS, shared prefixes, 9 sources, ..."""
    rng = random.Random(14)
    eng = engine_factory(8)
    twins = []
    big = FS_MAX_ITEMS + 3 if not EMUL else FS_MAX_ITEMS + 1
    for i in range(40):
        shape = i % 10
        mop = [COUNTER, UINT64ADD, APPEND, NONE][i % 4]
        t = engine_factory.twin(mop, wb=wb_for(big if shape == 2 else 3000, 3000 * 64))
        twins.append(t)
        pool = k16(rng, 600, prefix=bytes([0x10 + i]))
        if shape == 0:    # memtable only
            t.write(mixed_ops(rng, pool, rng.randint(1, 900), mop))
        elif shape == 1:  # runs only
            build_stack(t, rng, [300, 200], pool, mop)
        elif shape == 2:  # above the radix sort's limit
            t.write(mixed_ops(rng, keys_with_spread(rng, 20000, 40), big, mop, vlens=(8,)))
        elif shape == 3:  # shared prefixes (comparison sort)
            t.write(mixed_ops(rng, k16(rng, 900, prefix=b"PREFIX%02d" % i), 1500, mop))
        elif shape == 4:  # 9 sources
            build_stack(t, rng, [100, 150, 80, 120, 60, 90, 70], pool, mop)
            t.ingest(sorted((k, b"ingested") for k in set(rng.sample(pool, 100))))
            t.write(mixed_ops(rng, pool, 400, mop))
        elif shape == 5:  # one entry
            t.write([(T_PUT, pool[0], b"x")])
        elif shape == 6:  # a run and one tombstone
            build_stack(t, rng, [500], pool, mop)
            t.write([(T_DEL, pool[3], b"")])
        elif shape == 7:  # empty
            pass
        else:             # a few runs and a memtable, random sizes
            build_stack(t, rng, [rng.randint(1, 700) for _ in range(rng.randint(1, 5))], pool, mop)
            t.write(mixed_ops(rng, pool, rng.randint(1, 2500), mop))
    for name in ("flush_all", "compact_all"):
        ops = [Op(t) for t in twins]
        assert getattr(eng, name)() == OK
        for t, op in zip(twins, ops):
            bottom, _ = op.check()
            if name == "compact_all":
                assert bottom and len(dump_all(t.s)) <= 1
            check_reads(t, n_get=4)
        for t in twins[::3]:
            t.write(mixed_ops(rng, sorted(t.keys) or [b"k"], 200, t.merge_op))


# ---- background merges ---------------------------------------------------------------------------------------------
def test_background_merges_install_while_ticks_run(engine_factory):
    """background compaction on: merges install while ticks run; every run validated, every read against the oracle
    (which runs merge depends on timing, so no model here)"""
    rng = random.Random(15)
    eng = engine_factory(2, bg=True)
    twins = [engine_factory.twin(mop, wb=wb_for(3000, 3000 * 40)) for mop in (COUNTER, UINT64ADD, APPEND)]
    pools = [k16(rng, 500, prefix=bytes([0x20 + i])) for i in range(3)]
    for rnd in range(12):
        six, batches = [], []
        for i, t in enumerate(twins):
            for _ in range(3):
                ops = mixed_ops(rng, pools[i], 60, t.merge_op)
                t.keys.update(k for _, k, _ in ops)
                six.append(i)
                batches.append(batch_of(ops))
        st = eng.apply_many([twins[i].s.index for i in six], batches, [7] * len(batches))
        for i, b, st_ in zip(six, batches, st):
            assert twins[i].o.apply(b, 7) == st_ == OK
        for t in twins:
            if rnd % 2 == 0:
                assert t.s.flush() == OK
            validate_shard(t.s, merge_op=t.merge_op)
            check_reads(t, n_get=8)
    t0 = time.time()
    while sum(t.s.stats()["compactions"] for t in twins) == 0:
        assert time.time() - t0 < 120, "no background merge"
        time.sleep(0.02)
    for t in twins:
        validate_shard(t.s, merge_op=t.merge_op)
        check_reads(t)
