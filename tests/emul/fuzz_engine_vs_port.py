"""TEST INFRASTRUCTURE — differential fuzzer: the engine (compiled against the CPU emulation, tests/emul) against the
oracle port on random streams: every merge operator, variable and fixed key shapes, tiny and default write buffers
(forced flushes), flush / compaction at random points, single applies and multi-shard ticks (rsp_apply_many),
Get / MultiGet / full scans / iterator walks compared after every few batches, every run of a shard checked by
tests/test_compaction_gpu.py's validate_shard after each explicit flush and compaction.  GPU time is too scarce for hundreds of
seeds; the emulation runs them for free.  `python tests/emul/fuzz_engine_vs_port.py FIRST LAST [env VAR=1 ...]`.
A short range runs in tests/test_emul_cpu.py.
"""
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

from oracle import okv  # noqa: E402
from rocksplicator_b200 import engine  # noqa: E402
from streams import random_stream  # noqa: E402
from test_compaction_gpu import validate_shard  # noqa: E402


def iter_walk(db, keys, seed):
    rng = random.Random(seed)
    it = db.iterator()
    out = []
    for _ in range(24):
        r = rng.random()
        if r < 0.15:
            it.seek_to_first()
        elif r < 0.3:
            it.seek_to_last()
        elif r < 0.55:
            k = rng.choice(keys) if rng.random() < 0.7 else bytes(rng.getrandbits(8) for _ in range(rng.randint(0, 5)))
            it.seek(k)
        elif r < 0.8:
            if it.valid():
                it.next()
        else:
            if it.valid():
                it.prev()
        out.append((it.valid(), it.key() if it.valid() else None, it.value() if it.valid() else None, it.status()))
    it.close()
    return out


def compare(s, o, keys, tag):
    assert s.latest_seq() == o.latest_seq(), (tag, "seq", s.latest_seq(), o.latest_seq())
    probe = keys + [b"zz-missing", b""]
    assert s.multi_get(probe) == o.multi_get(probe), (tag, "multi_get")
    for k in probe[::5]:
        assert s.get(k) == o.get(k), (tag, "get", k)
    assert s.scan() == o.scan(), (tag, "scan")
    k16 = [k for k in keys if len(k) == 16]
    if k16:
        # the 16-byte-key kernels (k_multi_get16 / k_multi_get16d) through the fixed-shape entry point, hits and misses
        import numpy as np
        q = k16 + [bytes(15) + b"\x01", b"\xff" * 16]
        n = len(q)
        for stride in (64, 256):
            vals = np.zeros((n, stride), dtype=np.uint8)
            vlen = np.zeros(n, dtype=np.uint32)
            st = np.zeros(n, dtype=np.int32)
            rc = s.engine.multi_get_fixed(np.full(n, s.index, dtype=np.uint32), np.frombuffer(b"".join(q), dtype=np.uint8).copy(),
                                          16, vals, stride, vlen, st)
            assert rc == 0, (tag, "multi_get_fixed rc", rc)
            if stride == 64 and getattr(s, "fz_device_form", True):
                st, vlen, vals = device_multi_get(s, q, stride)   # same answers through the device-pointer form
            want = o.multi_get(q)
            for i in range(n):
                w_st, w_v = want[i]
                if w_st == 0 and len(w_v) > stride:
                    assert st[i] == 7 and vlen[i] == len(w_v), (tag, "fixed incomplete", i, st[i], vlen[i])
                else:
                    assert st[i] == w_st, (tag, "fixed st", i, int(st[i]), w_st)
                    if w_st == 0:
                        assert bytes(vals[i, :vlen[i]]) == w_v, (tag, "fixed value", i)
    assert iter_walk(s, keys, hash(tag) & 0xffff) == iter_walk(o, keys, hash(tag) & 0xffff), (tag, "iter")
    if getattr(s, "fz_device_form", True):
        # batched range scans (Seek + n x Next): entries equal the oracle iterator's; a failed merge on the way shows as
        # an empty value and the scan's status
        rng = random.Random(hash(tag) & 0xfff)
        starts = [rng.choice(keys) for _ in range(3)] + [b"", b"\xff\xff"]
        lim = rng.choice([1, 7, 40])
        res = s.engine.multi_scan([s.index] * len(starts), starts, lim, 1 << 20)
        for k0, (st_, recs) in zip(starts, res):
            it = o.iterator()
            it.seek(k0)
            want, wst = [], 0
            while it.valid() and len(want) < lim:
                want.append((it.key(), it.value()))
                wst = it.status()
                it.next()
            it.close()
            assert recs == want and st_ == wst, (tag, "multi_scan", k0, st_, wst, len(recs), len(want))


def staged_tick(eng, six, batches, ts):
    """the pre-staged form (what bench.py times): the batches go as one tick, or as two or three ticks that are all
    reserved and launched back to back before the first one's results are folded (in-flight reservations)"""
    import numpy as np
    n = len(batches)
    cuts = sorted(set(random.Random(n * 31 + len(batches[0])).sample(range(1, n), min(n - 1, random.Random(n).randint(0, 2))))) if n > 1 else []
    parts = [(a, b) for a, b in zip([0] + cuts, cuts + [n])]
    handles = [_stage(eng, six[a:b], batches[a:b], ts[a:b]) for a, b in parts]
    lib = eng.lib
    out = [None] * len(handles)
    launched = []

    def finish_launched():
        for j in launched:
            a, b = parts[j]
            st = np.zeros(b - a, dtype=np.int32)
            lib.rsp_apply_staged_finish(eng.h, handles[j], st.ctypes.data)
            out[j] = [int(x) for x in st]
        del launched[:]

    for j, h in enumerate(handles):
        rc = lib.rsp_reserve(eng.h, h)
        if rc == 11:  # Busy: a shard is full while earlier ticks are in flight — fold those first
            assert launched
            finish_launched()
            rc = lib.rsp_reserve(eng.h, h)
        assert rc == 0, rc
        assert lib.rsp_apply_staged_device(eng.h, h, None) == 0
        launched.append(j)
    finish_launched()
    for h in handles:
        lib.rsp_stage_free(h)
    return np.array([x for part in out for x in part], dtype=np.int32)


def _stage(eng, six, batches, ts):
    import ctypes as C
    import numpy as np
    n = len(batches)
    six = np.ascontiguousarray(six, dtype=np.uint32)
    off = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(np.fromiter((len(b) for b in batches), dtype=np.uint64, count=n), out=off[1:])
    blob = np.frombuffer(b"".join(batches) + b"\0", dtype=np.uint8).copy()
    tsa = np.ascontiguousarray(ts, dtype=np.uint64)
    h = C.c_void_p()
    lib = eng.lib
    assert lib.rsp_stage_build(eng.h, n, six.ctypes.data, blob.ctypes.data, off.ctypes.data, tsa.ctypes.data, C.byref(h)) == 0
    return h


def device_multi_get(s, q, stride):
    """rsp_multi_get_device with (emulated) device buffers: what bench.py's kernel-level phase calls"""
    import numpy as np
    n = len(q)
    six = np.full(n, s.index, dtype=np.uint32)
    keys = np.frombuffer(b"".join(q), dtype=np.uint8).copy()
    vals = np.zeros((n, stride), dtype=np.uint8)
    vlen = np.zeros(n, dtype=np.uint32)
    st = np.full(n, -1, dtype=np.int32)
    rc = s.engine.lib.rsp_multi_get_device(s.engine.h, n, six.ctypes.data, keys.ctypes.data, 16, vals.ctypes.data, stride,
                                           vlen.ctypes.data, st.ctypes.data, None)
    assert rc == 0
    return st, vlen, vals


def one_seed(eng, port, seed):
    rng = random.Random(seed * 7919 + 3)
    mop, mname = rng.choice([(okv.MERGE_COUNTER, "counter"), (okv.MERGE_APPEND, "append"),
                             (okv.MERGE_UINT64ADD, "counter"), (okv.MERGE_NONE, None)])
    bad = mop == okv.MERGE_COUNTER and rng.random() < 0.25
    n_shards = rng.choice([1, 1, 3])
    fixed = rng.random() < 0.35
    heavy = os.environ.get("FUZZ_HEAVY") == "1"  # longer streams over more keys, flushes twice as often
    keys, stream = random_stream(9000 + seed, rng.randint(300, 800) if heavy else rng.randint(20, 160),
                                 n_keys=rng.choice([200, 600]) if heavy else rng.choice([4, 12, 40, 90]), merge=mname,
                                 max_ops=rng.choice([1, 3, 8, 25]), var_len=not fixed, bad_operands=bad)
    if rng.random() < 0.3:
        # now and then a value far larger than the write buffer (the memtable has to be re-sized for the tick)
        from rocksplicator_b200.write_batch import WriteBatch
        for _ in range(rng.randint(1, 3)):
            big = WriteBatch().put(rng.choice(keys), rng.randbytes(rng.choice([5000, 70000, 300000])))
            if mname and rng.random() < 0.5:
                big.merge(rng.choice(keys), (8).to_bytes(8, "little") if mname == "counter" else b"+")
            stream.insert(rng.randrange(len(stream) + 1), (big.data(), rng.getrandbits(40)))
    wb = rng.choice([0, 0, 2048, 8192])
    shards = [eng.open_shard("fz%d_%d" % (seed, i), merge_op=mop, write_buffer_bytes=wb) for i in range(n_shards)]
    oracles = [okv.Okv(port, merge_op=mop) for _ in range(n_shards)]
    for s_ in shards:
        s_.fz_device_form = mop != okv.MERGE_APPEND  # the device form hands host-folded keys back (status 100)
    live = []  # iterators opened at some point and stepped while writes, flushes and compactions go on (snapshots)
    try:
        i = 0
        while i < len(stream):
            if n_shards > 1 or rng.random() < 0.3:
                # one tick for several batches over several shards; per-shard order == submission order
                m = min(len(stream) - i, rng.randint(1, 12))
                six = [rng.randrange(n_shards) for _ in range(m)]
                if rng.random() < 0.3:
                    st = staged_tick(eng, [shards[x].index for x in six], [stream[i + j][0] for j in range(m)],
                                     [stream[i + j][1] for j in range(m)])
                else:
                    st = eng.apply_many([shards[x].index for x in six], [stream[i + j][0] for j in range(m)],
                                        [stream[i + j][1] for j in range(m)])
                want = [oracles[six[j]].apply(stream[i + j][0], stream[i + j][1]) for j in range(m)]
                assert list(st) == want, (seed, i, list(st), want)
                i += m
            else:
                bt, ts = stream[i]
                if rng.random() < 0.25:
                    # the leader's entry point: the same walk without the follower's appended LogData(timestamp),
                    # which a well-formed batch does not notice
                    assert shards[0].write(bt) == oracles[0].apply(bt, ts), (seed, i, "write")
                else:
                    assert shards[0].apply(bt, ts) == oracles[0].apply(bt, ts), (seed, i)
                i += 1
            r = rng.random()
            x = rng.randrange(n_shards)
            if not bad:
                if r < (0.10 if heavy else 0.05):
                    shards[x].flush()
                    validate_shard(shards[x], merge_op=mop)
                elif r < (0.13 if heavy else 0.08):
                    shards[x].compact()
                    validate_shard(shards[x], merge_op=mop)
            if rng.random() < 0.08:
                compare(shards[x], oracles[x], keys, (seed, i, x))
            if rng.random() < 0.06 and len(live) < 6:
                ia, ib = shards[x].iterator(), oracles[x].iterator()
                if rng.random() < 0.5:
                    ia.seek_to_first(), ib.seek_to_first()
                else:
                    ia.seek_to_last(), ib.seek_to_last()
                live.append((ia, ib))
            for ia, ib in live:
                for _ in range(3):
                    got = (ia.valid(), ia.key() if ia.valid() else None, ia.value() if ia.valid() else None, ia.status())
                    want = (ib.valid(), ib.key() if ib.valid() else None, ib.value() if ib.valid() else None, ib.status())
                    assert got == want, (seed, i, "live iterator")
                    if ia.valid():
                        if rng.random() < 0.7:
                            ia.next(), ib.next()
                        else:
                            ia.prev(), ib.prev()
        if n_shards > 1:
            # one MultiGet call over a mix of shards (what a router fans in): any order, duplicates, misses
            pick = [(rng.randrange(n_shards), rng.choice(keys + [b"zz-missing"])) for _ in range(150)]
            got = eng.multi_get([shards[x].index for x, _ in pick], [k for _, k in pick])
            assert got == [oracles[x].get(k) for x, k in pick], (seed, "cross-shard multi_get")
        for x in range(n_shards):
            compare(shards[x], oracles[x], keys, (seed, "end", x))
            validate_shard(shards[x], merge_op=mop)
            if not bad:
                shards[x].compact()
                validate_shard(shards[x], merge_op=mop)
                compare(shards[x], oracles[x], keys, (seed, "compacted", x))
    finally:
        for ia, ib in live:
            ia.close(), ib.close()
        for s in shards:
            s.close()
        for o in oracles:
            o.close()


def run(first, last, lib_path, verbose=False):
    engine.SO_PATH = lib_path
    port = okv.load_port()
    eng = None
    bad = 0
    for seed in range(first, last):
        if eng is None or seed % 25 == 0:
            # a fresh engine now and then, with a different number of runs allowed to pile up before they are merged
            if eng is not None:
                eng.close()
            eng = engine.Engine(0, arena_bytes=1 << 24, l0_compaction_trigger=[0, 2, 8, 3][(seed // 25) % 4])
        try:
            one_seed(eng, port, seed)
        except AssertionError as ex:
            bad += 1
            print("DIVERGE seed", seed, str(ex)[:400])
        if verbose and seed % 10 == 9:
            print("seed", seed, "bad", bad, flush=True)
    eng.close()
    return bad


if __name__ == "__main__":
    lib = os.environ.get("RSP_TEST_EMUL_LIB", os.path.join(ROOT, "tests", "emul", "build", "librsp_b200_emul.so"))
    print("done bad=", run(int(sys.argv[1]), int(sys.argv[2]), lib, verbose=True))
