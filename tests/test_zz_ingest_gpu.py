"""GPU parity of rsp_ingest_sorted (DB::IngestExternalFile for a sorted set of Puts) against the reference's own RocksDB
ingesting the SAME file (written by rocksplicator_b200/sst.py; its answers recorded by oracle/gen_golden.py): contents,
reads and the sequence-number rules of rocksdb_replicator/tests/rocksdb_assumption_test.cpp:248-283.  Runs last (file
name) — it is the newest entry point.
"""
import os
import random

import pytest

import golden_util as G
from rocksplicator_b200 import sst
from rocksplicator_b200.write_batch import WriteBatch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from rocksplicator_b200 import engine
    e = engine.Engine(0)
    yield e
    e.close()


def _kv(n, seed, lo=0, hi=1 << 30, max_v=300):
    rnd = random.Random(seed)
    keys = sorted({b"k%012d" % rnd.randrange(lo, hi) for _ in range(n)})
    return [(k, rnd.randbytes(rnd.randrange(0, max_v))) for k in keys]


def ingest_inputs():
    """the files and WriteBatches of test_ingest_sequence_rules_and_contents, in the order they are applied"""
    f1 = _kv(3000, 1, lo=0, hi=1 << 20)
    wb1 = WriteBatch().put(f1[10][0], b"overwritten").delete(f1[11][0]).put(b"k-new", b"v").data()
    f2 = _kv(500, 2, lo=1 << 28, hi=1 << 29)
    f3 = sorted(dict([(k, b"third:" + v[:4]) for k, v in f1[::7]] + [(f1[11][0], b"back")]).items())
    f4 = [(f1[5][0], b"refused")]
    wb2 = WriteBatch().put(f3[0][0], b"after").delete(f2[0][0]).data()
    return f1, wb1, f2, f3, f4, wb2


class RecordedRef:
    """The reference's RocksDB given the same files (the bytes our writer produces) and WriteBatches: its answers, in
    call order, as oracle/gen_golden.py recorded them in tests/golden/differential.json"""

    def __init__(self):
        self.rec = iter(G.load("differential.json")["ingest_gpu"])

    def _next(self, kind, *inputs):
        r = next(self.rec)
        assert r[:len(inputs) + 1] == [kind, *inputs], (r, kind, inputs)
        return r[len(inputs) + 1:]

    def ingest(self, kv, allow=True):
        return self._next("ingest", G.sha256(sst.write_sst(kv)), int(allow))[0]

    def apply(self, batch, ts):
        return self._next("apply", G.sha256(batch), ts)[0]

    def check(self):
        """-> [latest_seq, digest of the full scan]"""
        return self._next("check")


def _check(s, want, seq, ref):
    assert s.latest_seq() == seq
    assert s.scan() == sorted(want.items())
    keys = list(want)[:: max(1, len(want) // 64)] + [b"k-absent", b"zzz"]
    got = s.multi_get(keys)
    assert got == [(0, want[k]) if k in want else (1, None) for k in keys]
    assert ref.check() == [seq, G.digest(sorted(want.items()))]


def test_ingest_sequence_rules_and_contents(eng):
    ref = RecordedRef()
    s = eng.open_shard("ingest-a")
    want = {}
    f1, wb1, f2, f3, f4, wb2 = ingest_inputs()
    # 1. into an empty shard: no sequence number is consumed
    assert s.ingest(f1) == 0
    assert ref.ingest(f1) == 0
    want.update(f1)
    _check(s, want, 0, ref)
    # 2. writes on top, then a file whose range lies beyond everything: still no bump
    assert s.apply(wb1, 1234) == 0
    assert ref.apply(wb1, 1234) == 0
    want[f1[10][0]] = b"overwritten"
    del want[f1[11][0]]
    want[b"k-new"] = b"v"
    _check(s, want, 3, ref)
    assert s.ingest(f2) == 0
    assert ref.ingest(f2) == 0
    want.update(f2)
    _check(s, want, 3, ref)
    # 3. an overlapping file is newer than everything and takes sequence number last+1
    assert s.ingest(f3) == 0
    assert ref.ingest(f3) == 0
    want.update(f3)
    _check(s, want, 4, ref)
    # 4. ... and is refused when global sequence numbers are not allowed; nothing changes
    assert s.ingest(f4, allow_global_seqno=False) == 4
    assert ref.ingest(f4, allow=False) != 0
    _check(s, want, 4, ref)
    # 5. later writes and a full compaction see the ingested data like any other
    assert s.apply(wb2, 1234) == 0
    assert ref.apply(wb2, 1234) == 0
    want[f3[0][0]] = b"after"
    del want[f2[0][0]]
    _check(s, want, 6, ref)
    assert s.compact() == 0
    _check(s, want, 6, ref)
    # 6. unsorted input: "Keys must be added in order"
    assert s.ingest([(b"b", b"1"), (b"a", b"2")]) == 4
    assert s.ingest([(b"a", b"1"), (b"a", b"2")]) == 4
    _check(s, want, 6, ref)
    s.close()
    assert next(ref.rec, None) is None


def test_ingest_fixed_shape_serves_the_fast_path(eng):
    """16 B keys / 64 B values (the bench shape): the ingested run carries the same hash index MultiGet16 uses"""
    import numpy as np
    from rocksplicator_b200 import synth
    n = 20000
    keys = synth.keys16(7, np.arange(n, dtype=np.uint64))
    vals = synth.values(7, 0, np.arange(n, dtype=np.uint64), 0, 64)
    kv = sorted((bytes(keys[i]), bytes(vals[i])) for i in range(n))
    s = eng.open_shard("ingest-b")
    assert s.ingest(kv) == 0 and s.latest_seq() == 0
    probe = [kv[i][0] for i in range(0, n, 37)] + [b"\xff" * 16]
    got = s.multi_get(probe)
    assert got[:-1] == [(0, kv[i][1]) for i in range(0, n, 37)] and got[-1] == (1, None)
    assert s.scan(limit=100) == kv[:100]
    s.close()


def test_gpudb_export_and_ingest_files():
    """GpuDB::ExportSstFile -> GpuDB::IngestExternalFile (tests/cpp/host_tests.cpp::test_gpu_export_and_ingest)"""
    import subprocess
    from rocksplicator_b200 import build
    _, exe = build.build_host()
    if os.environ.get("RSP_TEST_EMUL_LIB"):  # tests/test_emul_cpu.py: the same test binary linked against the emulation
        exe = os.path.join(os.path.dirname(os.environ["RSP_TEST_EMUL_LIB"]), "host_tests_emul")
    p = subprocess.run([exe, "gpu", "gpu_export_and_ingest"], capture_output=True, text=True, timeout=300)
    print(p.stdout[-4000:], p.stderr[-2000:])
    assert p.returncode == 0 and " 0 failures" in p.stdout and "[ RUN  ] gpu_export_and_ingest" in p.stdout, p.stdout[-3000:]
