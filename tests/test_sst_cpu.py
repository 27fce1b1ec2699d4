"""SST interchange on the host (SURVEY §8f rank 2), CPU only.
  * the reference's golden file rocksdb_admin/tests/old_sst_data.sst (copied byte-for-byte to tests/golden/: a 978-byte
    test fixture, Snappy-compressed block) must read as key0..key9 -> value0..value9 (sst_binary.cpp:43-58);
  * files written by the reference's own SstFileWriter (librocksdb.so.5.4, stored under tests/golden/) must read back
    exactly;
  * files written by OUR writer must be accepted by the reference's DB::IngestExternalFile and scan back exactly,
    with the sequence-number rule of rocksdb_assumption_test.cpp:248-262 (ingest into an empty DB: seq stays 0).
The reference's side of both was recorded by oracle/gen_golden.py."""
import os
import random
import tempfile

import pytest

import golden_util as G
from rocksplicator_b200 import sst

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN = os.path.join(GOLDEN_DIR, "old_sst_data.sst")
# (n, seed, max_v) of the files the reference wrote and tests/golden/ stores: the many-block file has short values to
# stay under 100 KB
REF_WRITTEN = ((1, 11, 2000), (50, 12, 2000), (2000, 13, 8))


def test_golden_old_sst_data():
    entries, props = sst.read_sst(open(GOLDEN, "rb").read())
    assert [(k, t, v) for k, _, t, v in entries] == [(b"key%d" % i, 1, b"value%d" % i) for i in range(10)]
    assert props["num_entries"] == 10
    assert all(seq == 0 for _, seq, _, _ in entries)


def test_rejects_garbage():
    with pytest.raises(ValueError):
        sst.read_sst(b"not an sst file at all, but long enough to have a footer ...............")
    data = bytearray(open(GOLDEN, "rb").read())
    data[10] ^= 0xFF  # flip a byte inside the first data block: the CRC32C must catch it
    with pytest.raises(ValueError):
        sst.read_sst(bytes(data))


def _kv(n, seed, max_v=300):
    rng = random.Random(seed)
    keys = sorted({bytes(rng.getrandbits(8) for _ in range(rng.randint(1, 40))) for _ in range(n)})
    return [(k, bytes(rng.getrandbits(8) for _ in range(rng.choice([0, 1, 8, 64, max_v])))) for k in keys]


def test_roundtrip_own_writer_reader():
    for n, seed in ((1, 1), (10, 2), (3000, 3)):
        kv = _kv(n, seed)
        entries, props = sst.read_sst(sst.write_sst(kv, block_size=512 if n > 100 else 4096))
        assert [(k, v) for k, _, _, v in entries] == kv
        assert props["external_version"] == 2 and props["num_entries"] == len(kv)
    with pytest.raises(ValueError):
        sst.write_sst([(b"b", b"1"), (b"a", b"2")])  # "Keys must be added in order"


def test_reads_files_written_by_the_reference():
    """tests/golden/ref_written_<n>.sst: what the reference's SstFileWriter wrote for _kv(n, seed, max_v)
    (oracle/gen_golden.py)"""
    for n, seed, max_v in REF_WRITTEN:
        kv = _kv(n, seed, max_v=max_v)
        entries, props = sst.read_sst(open(os.path.join(GOLDEN_DIR, "ref_written_%d.sst" % n), "rb").read())
        assert [(k, t, v) for k, _, t, v in entries] == [(k, 1, v) for k, v in kv]
        assert props["external_version"] == 2 and props["global_seqno"] == 0 and props["num_entries"] == len(kv)


def ingest_inputs(n, seed):
    """test_reference_ingests_files_written_here's two files: kv, then an overlapping update of every third key"""
    kv = _kv(n, seed, max_v=1500)
    return kv, [(k, b"second:" + v[:5]) for k, v in kv[::3]]


INGESTED = ((1, 21), (200, 22), (5000, 23))


def test_reference_ingests_files_written_here():
    """What the reference's DB::IngestExternalFile made of files written here, recorded by oracle/gen_golden.py in
    tests/golden/differential.json for these exact bytes (a writer that changes them has to be checked again)."""
    rec = G.load("differential.json")["sst_ingest"]
    for n, seed in INGESTED:
        kv, kv2 = ingest_inputs(n, seed)
        f1, f2 = sst.write_sst(kv), sst.write_sst(kv2)
        r = rec[str(n)]
        assert [r["file"], r["file2"]] == [G.sha256(f1), G.sha256(f2)], n
        assert r["rc"] == 0, r["error"]
        assert r["seq"] == 0  # ingest into an empty DB does not consume sequence numbers
        assert r["scan"] == G.digest(kv)
        assert r["get"] == G.digest([(0, v) for k, v in kv[:: max(1, len(kv) // 50)]])
        # an overlapping second ingest is given global sequence number last+1 (rocksdb_assumption_test.cpp:272-283)
        assert r["rc2"] == 0, r["error2"]
        assert r["seq2"] == 1
        want = dict(kv)
        want.update(kv2)
        assert r["scan2"] == G.digest(sorted(want.items()))
        # (move_files = false: RocksDB stamps the sequence number into ITS copy; the file written here is untouched)
        assert r["file2_after"] == G.sha256(f2)
        entries, props = sst.read_sst(f2)
        assert props["global_seqno"] == 0 and [(k, v) for k, _, _, v in entries] == kv2


def test_shard_file_helpers_host_half():
    """sst.export_file / sst.ingest_file around a stand-in shard: the file goes through the real writer and reader"""
    class Standin:
        def __init__(self, kv=()): self.kv = list(kv)
        def ingest(self, kv, allow_global_seqno=True): self.kv = list(kv); return 0
        def scan(self): return self.kv
    kv = _kv(300, 31)
    tmp = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    path = os.path.join(tmp, "shard.sst")
    assert sst.export_file(Standin(kv), path) == len(kv)
    dst = Standin()
    assert sst.ingest_file(dst, path) == 0 and dst.kv == kv
    # the reference's own golden file (SstFileWriter output, Snappy block) loads the same way
    assert sst.ingest_file(dst, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "old_sst_data.sst")) == 0
    assert dst.kv == [(b"key%d" % i, b"value%d" % i) for i in range(10)]
