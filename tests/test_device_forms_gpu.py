"""The device-pointer entry points (rsp_multi_get_device, rsp_multi_scan_device, rsp_stage_build -> rsp_reserve ->
rsp_apply_staged_device -> rsp_apply_staged_finish) against the oracle port, beyond the benchmark's shape.

These are the calls bench.py times, and the kernels behind them pick their code path from the buffers they are handed:
key / value pointer alignment, value stride, key length, number of runs, run size, merge operator.  Each case below
forces one of those paths and checks every answer in its raw device form (statuses, vlen markers, record bytes), with
a 0xA5 guard region around every output buffer that must come back untouched.

Device buffers are torch.cuda tensors, read back after a device synchronize.  Under the CPU emulation (tests/emul,
RSP_TEST_EMUL_LIB set) device memory is host memory: the buffers are numpy arrays and every stream is the engine's.
"""
import bisect
import os
import random
import struct
import time
from collections import defaultdict

import numpy as np
import pytest

from oracle import okv
from rocksplicator_b200.write_batch import WriteBatch
from streams import corrupt_cases, random_stream

pytestmark = pytest.mark.gpu

EMUL = bool(os.environ.get("RSP_TEST_EMUL_LIB"))
MAX_SHARDS = 64
PAD = 0xA5
GUARD = 64
OK, NOT_FOUND, INVALID_ARGUMENT, INCOMPLETE, BUSY = 0, 1, 4, 7, 11
HOST_MERGE = 100                 # d_st of a lookup / scan that needs the host-side merge operator
SCAN_TRUNCATED = 1 << 30         # scan status bit: a status was set AND the scan ran out of room
VLEN_HOST_FOLD, VLEN_MERGE_FAILED = 0xFFFFFFFF, 0xFFFFFFFE
MSG_OF_CODE = {2: 11, 4: 10}     # failed merge -> message id in the raw scan status (MSG_MERGE_FAILED / MSG_MERGE_NOT_INIT)
NONE, COUNTER, UINT64ADD, APPEND = okv.MERGE_NONE, okv.MERGE_COUNTER, okv.MERGE_UINT64ADD, okv.MERGE_APPEND
MERGE_NAMES = {NONE: "none", COUNTER: "counter", UINT64ADD: "uint64add", APPEND: "append"}


# ---- device buffers -------------------------------------------------------------------------------------------------
class Buf:
    """`n` bytes of device memory at byte `offset` past a 256-aligned base; everything around them is 0xA5."""

    def __init__(self, n, offset=0, data=None):
        self.n, self.offset = n, offset
        total = 256 + offset + n + GUARD
        if EMUL:
            self._raw = np.full(total, PAD, dtype=np.uint8)
            self._lo = (-self._raw.ctypes.data) % 256
            self.ptr = self._raw.ctypes.data + self._lo + offset
        else:
            import torch
            self._raw = torch.full((total,), PAD, dtype=torch.uint8, device="cuda")
            self._lo = (-self._raw.data_ptr()) % 256
            self.ptr = self._raw.data_ptr() + self._lo + offset
        if data is not None:
            assert len(data) == n
            a = self._lo + offset
            src = np.frombuffer(bytes(data), dtype=np.uint8)
            if EMUL:
                self._raw[a:a + n] = src
            elif n:
                import torch
                self._raw[a:a + n].copy_(torch.from_numpy(src.copy()))

    def read(self):
        """the n bytes (after sync()); asserts that the guard bytes before and after them are untouched"""
        r = self._raw[self._lo:] if EMUL else self._raw[self._lo:].cpu().numpy()
        r = np.array(r, copy=True)
        assert (r[:self.offset] == PAD).all() and (r[self.offset + self.n:] == PAD).all(), "write outside the buffer"
        return r[self.offset:self.offset + self.n]


def sync():
    if not EMUL:
        import torch
        torch.cuda.synchronize()


def caller_streams(k):
    """k streams other than the engine's (torch streams; the engine's own stream under the emulation)"""
    if EMUL:
        return [None] * k
    import torch
    return [torch.cuda.Stream() for _ in range(k)]


def handle(stream):
    return None if stream is None else stream.cuda_stream


# ---- engines and shards ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng():
    from rocksplicator_b200 import engine
    e = engine.Engine(0, max_shards=MAX_SHARDS)
    yield e
    e.close()


@pytest.fixture(scope="module")
def eng8():
    """runs pile up: a merge starts only at 8 runs"""
    from rocksplicator_b200 import engine
    e = engine.Engine(0, max_shards=MAX_SHARDS, l0_compaction_trigger=8)
    yield e
    e.close()


@pytest.fixture(scope="module")
def eng2():
    """background merges start at 2 runs"""
    from rocksplicator_b200 import engine
    e = engine.Engine(0, max_shards=MAX_SHARDS, l0_compaction_trigger=2)
    yield e
    e.close()


_n = [0]


def new_shard(eng, merge_op=NONE, **kw):
    _n[0] += 1
    return eng.open_shard("d%05d" % _n[0], merge_op=merge_op, **kw)


class Twin:
    """one engine shard and its oracle, written together; `opnd[k]`: the newest write of k is a Merge"""

    def __init__(self, eng, port, merge_op=NONE, **kw):
        self.eng, self.merge_op = eng, merge_op
        self.s = new_shard(eng, merge_op, **kw)
        self.o = okv.Okv(port, merge_op=merge_op)
        self.opnd = {}
        self._want = {}

    @property
    def index(self):
        return self.s.index

    def write(self, ops, ts=7):
        wb = WriteBatch()
        for op, k, *v in ops:
            getattr(wb, op)(k, *v)
            self.opnd[k] = op == "merge"
        d = wb.data()
        assert self.s.apply(d, ts) == 0 and self.o.apply(d, ts) == 0
        self._want.clear()

    def want_get(self, k):
        """what a device lookup of k answers: the oracle's Get, or HOST_MERGE for keys with operands under APPEND"""
        if k not in self._want:
            if self.merge_op == APPEND and self.opnd.get(k):
                self._want[k] = (HOST_MERGE, None)
            else:
                self._want[k] = self.o.get(k)
        return self._want[k]

    def close(self):
        self.s.close()
        self.o.close()


def make_keys(rng, n, klen, prefix=b""):
    """n distinct keys of klen bytes, last byte even (so that key + 1 in the last byte lies between two keys)"""
    out = set()
    while len(out) < n:
        out.add(prefix + rng.randbytes(klen - len(prefix) - 1) + bytes([2 * rng.randrange(128)]))
    return sorted(out)


def operand(rng, merge_op, i):
    if merge_op in (COUNTER, UINT64ADD):
        return b"bad" if merge_op == COUNTER and i % 23 == 0 else struct.pack("<q", rng.randint(-9, 9))
    return rng.randbytes(rng.choice([1, 8, 20]))


def churn(t, rng, keys, frac=0.4):
    """one round of overwrites, Deletes and Merges over a random part of the keys"""
    ops = []
    for i, k in enumerate(keys):
        if rng.random() >= frac:
            continue
        r = rng.random()
        if r < 0.4:
            ops.append(("put", k, rng.randbytes(rng.choice([8, 8, 64, 97, 300]))))
        elif r < 0.6:
            ops.append(("delete", k))
        else:
            ops.append(("merge", k, operand(rng, t.merge_op, i)))
    for i in range(0, len(ops), 50):
        t.write(ops[i:i + 50])


def wait_for_merge(t, timeout=120):
    t0 = time.time()
    while t.s.stats()["compactions"] == 0:
        assert time.time() - t0 < timeout, "no background merge"
        time.sleep(0.02)


# ---- rsp_multi_get_device -------------------------------------------------------------------------------------------
def build_get_state(eng, eng8, port, state, merge_op, klen, rng):
    keys = make_keys(rng, 240, klen)
    t = Twin(eng8 if state == "many_runs" else eng, port, merge_op)
    if state in ("fixed_run", "fixed_run_big"):  # (300-byte values: the 16-byte-key kernel's loop past 96 bytes)
        t.write([("put", k, rng.randbytes(300 if state == "fixed_run_big" else 64)) for k in keys])
        t.s.flush()
    elif state == "mixed_sizes":
        t.write([("put", k, rng.randbytes((0, 1, 96, 97, 300, 8)[i % 6])) for i, k in enumerate(keys)])
        t.s.flush()
    else:
        t.write([("put", k, rng.randbytes((8, 8, 64, 97)[i % 4])) for i, k in enumerate(keys)])
        if state == "memtable":
            t.s.flush()
            for _ in range(3):  # several versions per key in the memtable
                churn(t, rng, keys)
            assert t.s.stats()["memtable_entries"] > 0
        else:
            for _ in range(5 if state == "many_runs" else 6):
                t.s.flush()
                churn(t, rng, keys)
            t.s.flush()
            if state == "many_runs":
                assert t.s.stats()["n_runs"] >= 2
            else:
                wait_for_merge(t)
    return t, keys


def multi_get_buffers(six, keys, klen, stride, koff=0, voff=0):
    """inputs and outputs of one rsp_multi_get_device (sync() before the launch: the inputs are copied on torch's
    stream)"""
    n = len(keys)
    return {"six": Buf(4 * n, 0, np.asarray(six, dtype=np.uint32).tobytes()),
            "keys": Buf(n * klen, koff, b"".join(keys)),
            "vals": Buf(n * stride, voff), "vlen": Buf(4 * n), "st": Buf(4 * n), "n": n, "klen": klen, "stride": stride}


def launch_multi_get(eng, b, stream=None):
    rc = eng.lib.rsp_multi_get_device(eng.h, b["n"], b["six"].ptr, b["keys"].ptr, b["klen"], b["vals"].ptr, b["stride"],
                                      b["vlen"].ptr, b["st"].ptr, stream)
    assert rc == OK


def device_multi_get(eng, six, keys, klen, stride, koff=0, voff=0):
    """one rsp_multi_get_device on the engine's stream; returns the buffers (read them after sync())"""
    b = multi_get_buffers(six, keys, klen, stride, koff, voff)
    sync()
    launch_multi_get(eng, b)
    return b


def check_multi_get(b, who, keys, stride, tag):
    st = b["st"].read().view(np.int32)
    vlen = b["vlen"].read().view(np.uint32)
    vals = b["vals"].read().reshape(len(keys), stride)
    for i, (t, k) in enumerate(zip(who, keys)):
        at = (tag, i, k.hex(), int(st[i]), int(vlen[i]))
        if t is None:
            assert st[i] == INVALID_ARGUMENT, at
            continue
        w_st, w_v = t.want_get(k)
        if w_st == OK and len(w_v) > stride:
            assert st[i] == INCOMPLETE and vlen[i] == len(w_v), at
        else:
            assert st[i] == w_st, (at, w_st)
            if w_st == OK:
                assert vlen[i] == len(w_v) and vals[i, :vlen[i]].tobytes() == w_v, at


STRIDES = (8, 16, 64, 72, 128, 512)
GET_CASES = [
    ("fixed_run", NONE, 16), ("fixed_run", NONE, 8), ("fixed_run", NONE, 24), ("fixed_run_big", NONE, 16),
    ("mixed_sizes", NONE, 16), ("mixed_sizes", UINT64ADD, 24),
    ("memtable", NONE, 16), ("memtable", COUNTER, 16), ("memtable", UINT64ADD, 16), ("memtable", APPEND, 16),
    ("memtable", COUNTER, 8),
    ("many_runs", NONE, 16), ("many_runs", COUNTER, 16), ("many_runs", UINT64ADD, 16), ("many_runs", APPEND, 16),
    ("many_runs", UINT64ADD, 24),
    ("after_merge", COUNTER, 16), ("after_merge", APPEND, 16),
]


@pytest.mark.parametrize("state,merge_op,klen", GET_CASES,
                         ids=["%s-%s-k%d" % (s, MERGE_NAMES[m], k) for s, m, k in GET_CASES])
def test_multi_get_device(eng, eng8, port_lib, state, merge_op, klen):
    """every value stride (Incomplete at 8 / 16, unaligned 72, BIG 128 / 512), key pointer +8, value pointer +8;
    a second shard, a closed shard and ids >= max_shards mixed into the same launch in shuffled order, with duplicates"""
    rng = random.Random("%s/%d/%d" % (state, merge_op, klen))
    t, keys = build_get_state(eng, eng8, port_lib, state, merge_op, klen, rng)
    e = t.eng
    nb = Twin(e, port_lib)
    nb_keys = make_keys(rng, 40, klen)
    nb.write([("put", k, rng.randbytes(64)) for k in nb_keys])
    nb.s.flush()
    closed = new_shard(e)
    closed_ix = closed.index
    closed.close()
    try:
        misses = make_keys(rng, 12, klen) + [keys[5][:8] + bytes(klen - 8)]  # (shares the first 8 bytes of a key)
        look = [(t, k) for k in keys + misses] + [(nb, k) for k in nb_keys]
        look += [(None, k, ix) for ix, k in zip((closed_ix, MAX_SHARDS, 200, 0xFFFFFFFF), keys)]
        look += [rng.choice(look) for _ in range(60)]
        rng.shuffle(look)
        who = [x[0] for x in look]
        qk = [x[1] for x in look]
        six = [x[2] if x[0] is None else x[0].index for x in look]
        for stride in STRIDES:
            for koff, voff in ((0, 0), (8, 0), (0, 8)):
                b = device_multi_get(e, six, qk, klen, stride, koff, voff)
                sync()
                check_multi_get(b, who, qk, stride, (stride, koff, voff))
    finally:
        t.close()
        nb.close()


@pytest.fixture(scope="module")
def memtable_twin(eng, port_lib):
    rng = random.Random(4097)
    t, keys = build_get_state(eng, None, port_lib, "memtable", COUNTER, 16, rng)
    yield t, keys
    t.close()


@pytest.mark.parametrize("n", [1, 31, 33, 4097])
def test_multi_get_device_batch_sizes(eng, memtable_twin, n):
    t, keys = memtable_twin
    rng = random.Random(n)
    pool = [(t, k) for k in keys + make_keys(rng, 20, 16)] + [(None, keys[0])]
    look = [rng.choice(pool) for _ in range(n)]
    who = [x[0] for x in look]
    qk = [x[1] for x in look]
    six = [MAX_SHARDS + 3 if w is None else w.index for w in who]
    for stride, koff in ((64, 0), (72, 8)):
        b = device_multi_get(eng, six, qk, 16, stride, koff)
        sync()
        check_multi_get(b, who, qk, stride, (n, stride, koff))


def test_multi_get_device_two_streams_share_the_pending_list(eng, memtable_twin):
    """launches alternate between the engine's stream and two caller streams with nothing synchronized in between;
    every launch has its own buffers and lookups that leave the fast kernel (memtable versions, misaligned buffers)"""
    t, keys = memtable_twin
    rng = random.Random(2)
    s1, s2 = caller_streams(2)
    launches = []
    for j in range(9):
        koff, voff, stride = ((8, 0, 64), (0, 8, 64), (0, 0, 72))[j % 3]
        qk = [rng.choice(keys) for _ in range(rng.choice([33, 200, 500]))]
        launches.append((multi_get_buffers([t.index] * len(qk), qk, 16, stride, koff, voff), qk, stride))
    sync()
    for j, (b, _, _) in enumerate(launches):
        launch_multi_get(eng, b, handle((None, s1, s2)[(j + j // 3) % 3]))
    sync()
    for j, (b, qk, stride) in enumerate(launches):
        check_multi_get(b, [t] * len(qk), qk, stride, ("launch", j))


# ---- rsp_multi_scan_device ------------------------------------------------------------------------------------------
class ScanModel:
    """the shard's live entries in key order as the raw device scan reports them, taken from the oracle's iterator"""

    def __init__(self, t):
        self.t = t
        self.keys, self.recs, self.st = [], [], []
        it = t.o.iterator()
        it.seek_to_first()
        while it.valid():
            k, v, ist = it.key(), it.value(), it.status()
            if t.merge_op == APPEND and t.opnd.get(k):
                self.recs.append(struct.pack("<II", len(k), VLEN_HOST_FOLD) + k)
                self.st.append(HOST_MERGE)
            else:
                g_st, _ = t.o.get(k)
                if g_st != OK:  # a failed merge: the iterator shows the key with an empty value and raises its status
                    assert v == b"" and ist == g_st, (k.hex(), g_st, ist)
                    self.recs.append(struct.pack("<II", len(k), VLEN_MERGE_FAILED) + k)
                    self.st.append(g_st << 8 | MSG_OF_CODE[g_st])
                else:
                    self.recs.append(struct.pack("<II", len(k), len(v)) + k + v)
                    self.st.append(0)
            self.keys.append(k)
            it.next()
        it.close()

    def expect(self, start, max_entries, stride):
        """(st, n_out, bytes) of one scan"""
        i = bisect.bisect_left(self.keys, start)
        st, used, n = 0, 0, 0
        while n < max_entries and i + n < len(self.keys):
            r, rst = self.recs[i + n], self.st[i + n]
            if rst == HOST_MERGE:
                st = st or HOST_MERGE
            elif rst:
                st = rst
            if used + len(r) > stride:
                st = INCOMPLETE if st == 0 else st | SCAN_TRUNCATED
                break
            used += len(r)
            n += 1
        return st, n, b"".join(self.recs[i:i + n])

    def check_seek(self, start, max_entries):
        """the model against the oracle's own Seek + Next"""
        it = self.t.o.iterator()
        it.seek(start)
        i = bisect.bisect_left(self.keys, start)
        for j in range(min(max_entries, 130)):
            if not it.valid():
                assert i + j == len(self.keys)
                break
            assert it.key() == self.keys[i + j]
            it.next()
        it.close()


def build_scan_shard(eng, eng8, port, shape, rng):
    """-> (twin, key length, a few keys of the shard worth seeking to exactly)"""
    if shape.startswith("run_"):  # one run of that many 16/64 Puts
        n = int(shape[4:])
        t = Twin(eng, port, write_buffer_bytes=32 << 20)
        keys = make_keys(rng, n, 16)
        for i in range(0, n, 2000):
            t.write([("put", k, rng.randbytes(64)) for k in keys[i:i + 2000]])
        t.s.flush()
        st = t.s.stats()
        assert st["n_runs"] == 1 and st["run_entries"] == n
        return t, 16, [keys[0], keys[16383 if n > 16383 else n // 2], keys[n - 1], keys[n - 3]]
    if shape.startswith("runs_"):  # 2 .. 8 runs: overwrites, tombstones and merge operands across them
        merge_op = {"counter": COUNTER, "uint64add": UINT64ADD, "append": APPEND}[shape[5:]]
        t = Twin(eng8, port, merge_op)
        keys = make_keys(rng, 200, 16)
        t.write([("put", k, rng.randbytes((8, 8, 64, 97)[i % 4])) for i, k in enumerate(keys)])
        for _ in range(5):
            t.s.flush()
            churn(t, rng, keys)
        t.s.flush()
        assert t.s.stats()["n_runs"] >= 2
        return t, 16, [keys[0], keys[77], keys[-1]]
    if shape == "empty":
        return Twin(eng, port), 16, [bytes(15) + b"\x02"]
    klen, vlen, n, prefix = {"fast_16_64": (16, 64, 300, b""), "fast_32_8": (32, 8, 300, b""),
                             "general_24": (24, 64, 300, b""), "tombstones": (16, 64, 300, b""),
                             "shared_prefix_16": (16, 64, 3000, b"SAMEPFX!"),
                             "shared_prefix_24": (24, 40, 3000, b"SAMEPFX!")}[shape]
    t = Twin(eng, port)
    keys = make_keys(rng, n, klen, prefix)
    for i in range(0, n, 1000):
        t.write([("put", k, rng.randbytes(vlen)) for k in keys[i:i + 1000]])
    t.s.flush()
    if shape == "tombstones":  # a second run of Deletes (and a few overwrites) over the first
        t.write([("delete", k) for k in keys[::3]] + [("put", k, rng.randbytes(64)) for k in keys[1::7]])
        t.s.flush()
        assert t.s.stats()["n_runs"] == 2
    return t, klen, [keys[0], keys[n // 2], keys[-1]]


SCAN_SHAPES = ["fast_16_64", "fast_32_8", "general_24", "tombstones", "runs_counter", "runs_uint64add", "runs_append",
               "run_16384", "run_16385", "run_40000", "shared_prefix_16", "shared_prefix_24", "empty"]


def device_scan(eng, six, starts, klen, max_entries, stride, ooff=0):
    n = len(starts)
    b = {"six": Buf(4 * n, 0, np.asarray(six, dtype=np.uint32).tobytes()),
         "keys": Buf(n * klen, 0, b"".join(starts)),
         "out": Buf(n * stride, ooff), "n_out": Buf(4 * n), "st": Buf(4 * n)}
    sync()
    rc = eng.lib.rsp_multi_scan_device(eng.h, n, b["six"].ptr, b["keys"].ptr, klen, max_entries, b["out"].ptr, stride,
                                       b["n_out"].ptr, b["st"].ptr, None)
    assert rc == OK
    sync()
    return b["out"].read(), b["n_out"].read().view(np.uint32), b["st"].read().view(np.int32)


def check_scan(model, six, starts, max_entries, stride, got, tag):
    out, n_out, st = got
    for i, (ix, k) in enumerate(zip(six, starts)):
        slot = out[i * stride:(i + 1) * stride]
        at = (tag, i, k.hex(), int(st[i]), int(n_out[i]))
        if ix != model.t.index:
            assert st[i] == INVALID_ARGUMENT and n_out[i] == 0 and (slot == PAD).all(), at
            continue
        w_st, w_n, w_bytes = model.expect(k, max_entries, stride)
        assert (st[i], n_out[i]) == (w_st, w_n), (at, w_st, w_n)
        assert slot[:len(w_bytes)].tobytes() == w_bytes, at
        assert (slot[len(w_bytes):] == PAD).all(), (at, "bytes written past the last record")


@pytest.mark.parametrize("shape", SCAN_SHAPES)
def test_multi_scan_device(eng, eng8, port_lib, shape):
    """Seek before the first key, to an exact key, between two keys and past the last key; max_entries 0, 1, 7, 128 and
    more than the shard holds; roomy, exact-fit and short output strides, output at +4; unknown and closed shards in
    the same launch (7 scans: not a multiple of the kernel's 4 warps per block)"""
    rng = random.Random(shape)
    t, klen, exact = build_scan_shard(eng, eng8, port_lib, shape, rng)
    e = t.eng
    closed = new_shard(e)
    closed_ix = closed.index
    closed.close()
    try:
        e.flush_all()
        model = ScanModel(t)
        between = [k[:-1] + bytes([k[-1] + 1]) for k in exact[1:2]]
        starts = [bytes(klen)] + exact + between + [b"\xff" * klen]
        mixed_six = [t.index] * len(starts) + [MAX_SHARDS, closed_ix, 200]
        mixed = starts + [starts[1]] * 3
        if len(mixed) % 4 == 0:
            mixed_six, mixed = mixed_six[:-1], mixed[:-1]
        total = len(model.keys)
        for max_entries in (0, 1, 7, 128, total + 5):
            for k in starts:
                model.check_seek(k, max_entries)
            need = [len(model.expect(k, max_entries, 1 << 62)[2]) for k in starts]
            roomy = (max(need) + 16 + 7) // 8 * 8
            first = None
            for ooff in (0, 4):  # +4 takes the output out of the fast path's reach: same answers
                got = device_scan(e, mixed_six, mixed, klen, max_entries, roomy, ooff)
                check_scan(model, mixed_six, mixed, max_entries, roomy, got, (max_entries, "roomy", ooff))
                if first is None:
                    first = got
                else:
                    assert all((a == b).all() for a, b in zip(first, got))
            if total > 20000 and max_entries > 128 and EMUL:
                continue  # (exact fits of a 40,000-entry scan: the GPU run has them; the emulation is too slow)
            for k, nd in zip(starts, need):
                for stride in sorted({nd, nd - 1, nd - 8, nd - 88} & set(range(0, nd + 1))):
                    got = device_scan(e, [t.index], [k], klen, max_entries, stride)
                    check_scan(model, [t.index], [k], max_entries, stride, got, (max_entries, stride, k.hex()))
    finally:
        t.close()


def test_multi_scan_device_raw_statuses(eng, port_lib):
    """the raw contract on hand-made shards: a failed COUNTER merge -> vlen 0xfffffffe and st >> 8 == the oracle's
    status; APPEND operands -> vlen 0xffffffff and st == 100; running out of room after either sets bit 30"""
    for merge_op in (COUNTER, APPEND):
        t = Twin(eng, port_lib, merge_op)
        try:
            keys = [b"key-%012d" % i for i in range(8)]
            t.write([("put", k, struct.pack("<q", i)) for i, k in enumerate(keys)])
            t.s.flush()
            t.write([("merge", keys[2], b"bad" if merge_op == COUNTER else b"+x"), ("put", keys[5], b"v" * 40)])
            t.s.flush()
            eng.flush_all()
            model = ScanModel(t)
            assert model.st[2] == (2 << 8 | 11 if merge_op == COUNTER else HOST_MERGE)
            start = bytes(16)
            for max_entries, stride, want_st in ((8, 4096, model.st[2]), (2, 4096, 0),
                                                 (8, 3 * 24 + 8, model.st[2] | SCAN_TRUNCATED),
                                                 (8, 2 * 24, INCOMPLETE)):
                got = device_scan(eng, [t.index], [start], 16, max_entries, stride)
                assert got[2][0] == want_st, (merge_op, max_entries, stride, int(got[2][0]))
                check_scan(model, [t.index], [start], max_entries, stride, got, (merge_op, max_entries, stride))
        finally:
            t.close()


# ---- staged ticks ---------------------------------------------------------------------------------------------------
def stage(eng, items):
    """items: [(twin, batch bytes, ts)] -> rsp_staged*"""
    import ctypes as C
    n = len(items)
    six = np.array([t.index for t, _, _ in items], dtype=np.uint32)
    off = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(np.fromiter((len(b) for _, b, _ in items), dtype=np.uint64, count=n), out=off[1:])
    blob = np.frombuffer(b"".join(b for _, b, _ in items) + b"\0", dtype=np.uint8).copy()
    ts = np.array([x for _, _, x in items], dtype=np.uint64)
    h = C.c_void_p()
    assert eng.lib.rsp_stage_build(eng.h, n, six.ctypes.data, blob.ctypes.data, off.ctypes.data, ts.ctypes.data,
                                   C.byref(h)) == OK
    return h


def run_ticks(eng, ticks, depth, streams):
    """reserve and launch up to `depth` ticks before the oldest is folded; Busy from rsp_reserve folds the ticks in
    flight and retries.  A round of ticks in flight shares one stream; the next round takes the next stream.  Every
    fold is checked against the oracle, batch by batch.  Returns how often rsp_reserve answered Busy."""
    handles = [stage(eng, items) for items in ticks]
    lib = eng.lib
    in_flight, busy, rounds = [], 0, 0

    def fold_all():
        for j in in_flight:
            st = np.full(len(ticks[j]), -1, dtype=np.int32)
            rc = lib.rsp_apply_staged_finish(eng.h, handles[j], st.ctypes.data)
            want = [t.o.apply(b, ts) for t, b, ts in ticks[j]]
            assert list(st) == want, ("tick", j, list(st), want)
            assert rc in want if any(want) else rc == OK, ("tick", j, rc)  # (the status of a failing batch)
        del in_flight[:]

    try:
        for j, h in enumerate(handles):
            rc = lib.rsp_reserve(eng.h, h)
            if rc == BUSY:
                assert in_flight
                busy += 1
                fold_all()
                rounds += 1
                rc = lib.rsp_reserve(eng.h, h)
            assert rc == OK, rc
            assert lib.rsp_apply_staged_device(eng.h, h, handle(streams[rounds % len(streams)])) == OK
            in_flight.append(j)
            if len(in_flight) == depth:
                fold_all()
                rounds += 1
        fold_all()
    finally:
        for h in handles:
            lib.rsp_stage_free(h)
    return busy


def check_final(twins, keys):
    for t in twins:
        assert t.s.latest_seq() == t.o.latest_seq()
        assert t.s.scan() == t.o.scan()
        probe = keys + [b"zz-missing"]
        assert t.s.multi_get(probe) == t.o.multi_get(probe)


def interleave(rng, seqs):
    """one list of the sequences' items, each sequence's order kept, sequences mixed at random"""
    pos = [0] * len(seqs)
    out = []
    while True:
        live = [i for i, s in enumerate(seqs) if pos[i] < len(s)]
        if not live:
            return out
        i = rng.choice(live)
        out.append(seqs[i][pos[i]])
        pos[i] += 1


def cut(rng, items, lo, hi):
    out, i = [], 0
    while i < len(items):
        m = rng.randint(lo, hi)
        out.append(items[i:i + m])
        i += m
    return out


TICK_CASES = ["multi_op_interleaved", "long_groups_chunks", "large_batches_general", "busy_retry", "background_merges"]


@pytest.mark.parametrize("case", TICK_CASES)
def test_staged_ticks(eng, eng2, port_lib, case):
    rng = random.Random(case)
    streams = [None] + caller_streams(1)
    twins, keys = [], []
    try:
        if case == "multi_op_interleaved":
            # Put / Merge / Delete / SingleDelete / LogData batches for four merge operators, shards interleaved, a
            # corrupt batch in the middle of one shard's sequence (its error latches for the rest of it)
            seqs = []
            for i, (mop, mname) in enumerate(((COUNTER, "counter"), (UINT64ADD, "counter"), (NONE, None),
                                              (APPEND, "append"))):
                t = Twin(eng, port_lib, mop)
                twins.append(t)
                ks, stream = random_stream(700 + i, 40, n_keys=30, merge=mname, max_ops=8, var_len=True,
                                           bad_operands=mop == COUNTER)
                keys += ks
                items = [(t, b, ts) for b, ts in stream]
                if i == 1:
                    items.insert(20, (t, dict(corrupt_cases())["count_high"], 5))
                seqs.append(items)
            ticks = cut(rng, interleave(rng, seqs), 5, 30)
            depth = 3
        elif case == "long_groups_chunks":
            # more than 64 batches of one shard in a tick and batches over 4 KB: k_tick_chunks
            for i in range(2):
                twins.append(Twin(eng, port_lib, UINT64ADD))
            keys = [b"lg-%04d" % i for i in range(90)]
            seqs = [[(t, WriteBatch().put(rng.choice(keys), rng.randbytes(5000 if j % 9 == 0 else 40))
                      .merge(rng.choice(keys), struct.pack("<Q", j)).data(), j) for j in range(200)] for t in twins]
            ticks = [interleave(rng, [s[:150] for s in seqs]), interleave(rng, [s[150:] for s in seqs])]
            depth = 2
        elif case == "large_batches_general":
            # batches over 16 KB: the decode / sequence / insert / publish kernels
            twins.append(Twin(eng, port_lib, COUNTER))
            twins.append(Twin(eng, port_lib, NONE))
            keys = [b"lb-%03d" % i for i in range(40)]
            items = []
            for j in range(24):
                t = twins[j % 2]
                wb = WriteBatch().put(rng.choice(keys), rng.randbytes(17000 if j % 3 == 0 else 100))
                wb.delete(rng.choice(keys)).merge(rng.choice(keys), struct.pack("<q", j)).put_log_data(b"x" * 9)
                items.append((t, wb.data(), j))
            ticks = cut(rng, items, 3, 8)
            depth = 3
        elif case == "busy_retry":
            # an 8 KB memtable: a reservation while earlier ticks are in flight finds the shard full
            twins.append(Twin(eng, port_lib, COUNTER, write_buffer_bytes=8192))
            keys = [b"bz-%03d" % i for i in range(60)]
            items = [(twins[0], WriteBatch().put(rng.choice(keys), rng.randbytes(200))
                      .merge(rng.choice(keys), struct.pack("<q", j)).data(), j) for j in range(240)]
            ticks = cut(rng, items, 8, 12)
            depth = 4
        else:
            # l0_compaction_trigger=2 and small memtables: flushes on the reserve path, merges installed by the
            # background thread while ticks are in flight (they must keep the device's sequencing state)
            for mop in (COUNTER, NONE):
                twins.append(Twin(eng2, port_lib, mop, write_buffer_bytes=16384))
            keys = [b"bg-%03d" % i for i in range(80)]
            items = [(twins[j % 2], WriteBatch().put(rng.choice(keys), rng.randbytes(rng.choice([8, 100, 300])))
                      .delete(rng.choice(keys)).data(), j) for j in range(800)]
            ticks = cut(rng, items, 10, 20)
            depth = 3
        busy = run_ticks(eng2 if case == "background_merges" else eng, ticks, depth, streams)
        if case == "busy_retry":
            assert busy > 0
        if case == "background_merges":
            for t in twins:
                wait_for_merge(t)
        check_final(twins, keys)
    finally:
        for t in twins:
            t.close()


def test_reads_beside_ticks(eng, port_lib):
    """staged ticks on the engine's stream while device MultiGets run on a caller stream, over a shard with a memtable
    and two runs: every answer is a version of its key the oracle saw; once synchronized, the final state"""
    rng = random.Random(3)
    t = Twin(eng, port_lib)
    try:
        keys = make_keys(rng, 256, 16)
        versions = defaultdict(set)
        for _ in range(2):
            vals = [rng.randbytes(64) for _ in keys]
            t.write([("put", k, v) for k, v in zip(keys, vals)])
            for k, v in zip(keys, vals):
                versions[k].add(v)
            t.s.flush()
        vals = [rng.randbytes(64) for _ in keys[::2]]
        t.write([("put", k, v) for k, v in zip(keys[::2], vals)])
        for k, v in zip(keys[::2], vals):
            versions[k].add(v)
        ticks = []
        for j in range(8):
            items = []
            for _ in range(64):
                k, v = rng.choice(keys), rng.randbytes(64)
                versions[k].add(v)
                items.append((t, WriteBatch().put(k, v).data(), j))
            ticks.append(items)
        handles = [stage(eng, items) for items in ticks]
        (reader,) = caller_streams(1)
        reads = []
        for _ in ticks:
            qk = [rng.choice(keys) for _ in range(300)]
            reads.append((multi_get_buffers([t.index] * len(qk), qk, 16, 64), qk))
        sync()
        in_flight = []
        lib = eng.lib
        try:
            for j, h in enumerate(handles):
                assert lib.rsp_reserve(eng.h, h) == OK
                assert lib.rsp_apply_staged_device(eng.h, h, None) == OK
                in_flight.append(j)
                launch_multi_get(eng, reads[j][0], handle(reader))
                if len(in_flight) == 2:
                    j0 = in_flight.pop(0)
                    st = np.full(len(ticks[j0]), -1, dtype=np.int32)
                    assert lib.rsp_apply_staged_finish(eng.h, handles[j0], st.ctypes.data) == OK
                    assert list(st) == [t.o.apply(b, ts) for _, b, ts in ticks[j0]]
            for j0 in in_flight:
                st = np.full(len(ticks[j0]), -1, dtype=np.int32)
                assert lib.rsp_apply_staged_finish(eng.h, handles[j0], st.ctypes.data) == OK
                assert list(st) == [t.o.apply(b, ts) for _, b, ts in ticks[j0]]
        finally:
            for h in handles:
                lib.rsp_stage_free(h)
        sync()
        for r, (b, qk) in enumerate(reads):
            st = b["st"].read().view(np.int32)
            vlen = b["vlen"].read().view(np.uint32)
            vals = b["vals"].read().reshape(len(qk), 64)
            for i, k in enumerate(qk):
                assert st[i] == OK and vlen[i] == 64 and vals[i].tobytes() in versions[k], (r, i)
        assert t.s.latest_seq() == t.o.latest_seq()
        b = device_multi_get(eng, [t.index] * len(keys), keys, 16, 64)
        sync()
        check_multi_get(b, [t] * len(keys), keys, 64, "final")
    finally:
        t.close()
