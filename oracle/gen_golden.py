"""Generate tests/golden/*.json and tests/golden/ref_written_*.sst from the reference's OWN RocksDB binary (oracle/_ref).

Needs oracle/_ref, which `make -C oracle ref` builds from the reference's sources:
    python -m oracle.gen_golden
The fixtures pin the oracle port (tests/test_oracle_golden.py), the SST reader / writer (tests/test_sst_cpu.py) and the
CUDA engine (tests/test_parity_gpu.py, tests/test_zz_ingest_gpu.py) to outputs of the reference itself, so the tests
need neither the reference nor its binary.
TEST INFRASTRUCTURE ONLY.
"""
import ctypes as C
import json
import os
import shutil
import struct
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import okv  # noqa: E402
from golden_util import digest, sha256  # noqa: E402
from streams import corrupt_cases, random_stream  # noqa: E402
from rocksplicator_b200 import sst  # noqa: E402
from rocksplicator_b200.write_batch import WriteBatch  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
MERGES = {"none": okv.MERGE_NONE, "counter": okv.MERGE_COUNTER, "uint64add": okv.MERGE_UINT64ADD,
          "append": okv.MERGE_APPEND}


def snapshot(db, keys):
    """Everything the read path can observe: seq, per-key Get, MultiGet (with duplicates + a miss),
    forward scan, backward scan, a few Seeks."""
    probe = list(keys) + [b"zz-missing"] + list(keys[:3])
    it = db.iterator()
    it.seek_to_last()
    rev = []
    while it.valid():
        rev.append([it.key().hex(), it.value().hex()])
        it.prev()
    seeks = []
    for k in list(keys[:8]) + [b"", b"\x00", b"m", b"\xff\xff"]:
        it.seek(k)
        seeks.append([k.hex(), [it.key().hex(), it.value().hex()] if it.valid() else None])
    st = it.status()
    it.close()
    return {
        "seq": db.latest_seq(),
        "get": [[k.hex(), rc, v.hex() if v is not None else None] for k in probe for rc, v in [db.get(k)]],
        "multi_get": [[rc, v.hex() if v is not None else None] for rc, v in db.multi_get(probe)],
        "scan": [[k.hex(), v.hex()] for k, v in db.scan()],
        "rscan": rev,
        "seek": seeks,
        "iter_status": st,
    }


def gen_streams(ref):
    cases = []
    for merge in ("counter", "append", "uint64add", "none"):
        for seed in range(3):
            bad = merge == "counter" and seed == 2
            keys, stream = random_stream(1000 + 17 * seed + MERGES[merge], 60, n_keys=24,
                                         merge=None if merge == "none" else ("counter" if merge == "uint64add" else merge),
                                         bad_operands=bad)
            db = okv.Okv(ref, merge_op=MERGES[merge])
            steps = []
            for i, (b, ts) in enumerate(stream):
                rc = db.apply(b, ts)
                steps.append({"batch": b.hex(), "ts": ts, "rc": rc, "seq": db.latest_seq()})
                if i == 29 and not bad:
                    db.flush()
            mid = None
            if not bad:
                db.compact()
            final = snapshot(db, keys)
            db.close()
            cases.append({"name": f"{merge}-{seed}", "merge": merge, "keys": [k.hex() for k in keys],
                          "steps": steps, "final": final, "mid": mid})
    return cases


def gen_corrupt(ref):
    out = []
    pre = WriteBatch().put(b"pre", b"x").data()
    for name, b in corrupt_cases():
        db = okv.Okv(ref, merge_op=okv.MERGE_UINT64ADD)
        assert db.apply(pre, 1) == 0
        rc = db.apply(b, 0x1122334455667788)
        msg = db.last_error
        seq = db.latest_seq()
        rc2 = db.apply(pre, 2)  # the error latch (SURVEY §9 row 20)
        out.append({"name": name, "batch": b.hex(), "rc": rc, "msg": msg, "seq": seq, "rc_after": rc2,
                    "msg_after": db.last_error, "seq_after": db.latest_seq(),
                    "scan": [[k.hex(), v.hex()] for k, v in db.scan()]})
        db.close()
    return out


def gen_known_answers(ref):
    """SURVEY §9 rows 1-13 replayed on the binary (known-answer table)."""
    u64 = lambda x: struct.pack("<Q", x)  # noqa: E731
    rows = []
    db = okv.Okv(ref, merge_op=okv.MERGE_UINT64ADD)
    rows.append(["fresh_seq", db.latest_seq()])
    b = WriteBatch().put(b"k1", b"v1").delete(b"k2").merge(b"c", u64(5)).put_log_data(u64(1234)).set_sequence(999)
    rows.append(["row2_rc", db.apply(b.data(), 5)])
    rows.append(["row2_seq", db.latest_seq()])
    rows.append(["row3_rc", db.apply(WriteBatch().put_log_data(u64(1)).data(), 5)])
    rows.append(["row3_seq", db.latest_seq()])
    rows.append(["row4_rc", db.apply(bytes(12), 5)])
    rows.append(["row4_seq", db.latest_seq()])
    db.apply(WriteBatch().merge(b"c", u64(7)).data(), 5)
    rows.append(["row5_get_c", db.get(b"c")[1].hex()])
    db.apply(WriteBatch().merge(b"k1", u64(1)).data(), 5)
    rows.append(["row6_get_k1", db.get(b"k1")[1].hex()])
    db.apply(WriteBatch().put(b"z", u64(100)).delete(b"z").merge(b"z", u64(3)).merge(b"z", u64(4)).data(), 5)
    rows.append(["row7_seq", db.latest_seq()])
    rows.append(["row7_get_z", db.get(b"z")[1].hex()])
    db.apply(WriteBatch().put(b"x", b"1").put(b"x", b"2").delete(b"x").put(b"x", b"3").delete(b"y").data(), 5)
    rows.append(["row8_seq", db.latest_seq()])
    rows.append(["row8_get_x", db.get(b"x")[1].hex()])
    rows.append(["row8_get_y_rc", db.get(b"y")[0]])
    db.apply(WriteBatch().put(b"", b"").put(b"ev", b"").data(), 5)
    rows.append(["row9_get_empty", list(db.get(b""))[0], db.get(b"")[1].hex()])
    rows.append(["row10_scan", [[k.hex(), v.hex()] for k, v in db.scan()]])
    rows.append(["row10_seek_k", [[k.hex(), v.hex()] for k, v in db.scan(start=b"k", limit=1)]])
    rows.append(["row11_multi_get", [[rc, v.hex() if v is not None else None]
                                     for rc, v in db.multi_get([b"c", b"zz", b"c", b"k2", b"ev", b""])]])
    db.flush()
    rows.append(["row12_scan_after_flush", [[k.hex(), v.hex()] for k, v in db.scan()]])
    rows.append(["row12_seq", db.latest_seq()])
    db.apply(WriteBatch().single_delete(b"ev").data(), 5)
    rows.append(["row18_seq", db.latest_seq()])
    rows.append(["row18_get_ev_rc", db.get(b"ev")[0]])
    db.close()
    db = okv.Okv(ref, merge_op=okv.MERGE_NONE)
    rows.append(["row13_write_rc", db.apply(WriteBatch().merge(b"m", b"1").data(), 5)])
    rows.append(["row13_seq", db.latest_seq()])
    rc, _ = db.get(b"m")
    rows.append(["row13_get_rc", rc, db.last_error])
    db.close()
    return rows


def _sst_api(ref):
    ref.okv_write_sst.restype = C.c_int
    ref.okv_write_sst.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_void_p, C.c_char_p, C.c_void_p, C.c_char_p, C.c_size_t]
    ref.okv_ingest_sst.restype = C.c_int
    ref.okv_ingest_sst.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_char_p, C.c_size_t]


def _ingest(ref, db, tmp, data, allow=True):
    """-> (rc, error text, path of the ingested file)"""
    path = os.path.join(tmp, "f%d.sst" % len(os.listdir(tmp)))
    with open(path, "wb") as f:
        f.write(data)
    err = C.create_string_buffer(256)
    rc = ref.okv_ingest_sst(db.h, path.encode(), 1 if allow else 0, err, 256)
    return rc, err.value.decode(), path


def gen_ref_written(ref):
    """tests/golden/ref_written_<n>.sst: the reference's SstFileWriter on test_sst_cpu.REF_WRITTEN"""
    import numpy as np
    from test_sst_cpu import REF_WRITTEN, _kv
    for n, seed, max_v in REF_WRITTEN:
        kv = _kv(n, seed, max_v=max_v)
        koff = np.zeros(len(kv) + 1, dtype=np.uint64)
        voff = np.zeros(len(kv) + 1, dtype=np.uint64)
        np.cumsum([len(k) for k, _ in kv], out=koff[1:])
        np.cumsum([len(v) for _, v in kv], out=voff[1:])
        path = os.path.join(OUT, "ref_written_%d.sst" % n)
        err = C.create_string_buffer(256)
        rc = ref.okv_write_sst(path.encode(), len(kv), b"".join(k for k, _ in kv) + b"\0", koff.ctypes.data,
                               b"".join(v for _, v in kv) + b"\0", voff.ctypes.data, err, 256)
        assert rc == 0, err.value
        print(os.path.basename(path), os.path.getsize(path), "bytes")


def gen_sst_ingest(ref, tmp):
    """test_sst_cpu.test_reference_ingests_files_written_here: the reference ingesting the files our writer produces"""
    from test_sst_cpu import INGESTED, ingest_inputs
    out = {}
    for n, seed in INGESTED:
        kv, kv2 = ingest_inputs(n, seed)
        f1, f2 = sst.write_sst(kv), sst.write_sst(kv2)
        db = okv.Okv(ref)
        rc, error, _ = _ingest(ref, db, tmp, f1)
        r = {"file": sha256(f1), "rc": rc, "error": error, "seq": db.latest_seq(), "scan": digest(db.scan()),
             "get": digest([db.get(k) for k, _ in kv[:: max(1, len(kv) // 50)]])}
        rc, error, path2 = _ingest(ref, db, tmp, f2)
        with open(path2, "rb") as f:
            after = f.read()
        r.update({"file2": sha256(f2), "rc2": rc, "error2": error, "seq2": db.latest_seq(), "scan2": digest(db.scan()),
                  "file2_after": sha256(after)})
        db.close()
        out[str(n)] = r
    return out


def gen_ingest_gpu(ref, tmp):
    """test_zz_ingest_gpu.test_ingest_sequence_rules_and_contents: the reference's answers, call by call (RecordedRef)"""
    from test_zz_ingest_gpu import ingest_inputs
    f1, wb1, f2, f3, f4, wb2 = ingest_inputs()
    db = okv.Okv(ref)
    out = []

    def ingest(kv, allow=True):
        data = sst.write_sst(kv)
        out.append(["ingest", sha256(data), int(allow), _ingest(ref, db, tmp, data, allow)[0]])

    def apply(batch):
        out.append(["apply", sha256(batch), 1234, db.apply(batch, 1234)])

    def check():
        out.append(["check", db.latest_seq(), digest(db.scan())])

    ingest(f1), check()
    apply(wb1), check()
    ingest(f2), check()
    ingest(f3), check()
    ingest(f4, allow=False), check()
    apply(wb2), check()
    check()  # after the shard's full compaction
    check()  # after the two unsorted files it refuses
    db.close()
    return out


def gen_differential(ref):
    """The reference's side of the differential tests, as digests (golden_util.digest) of what it returned"""
    from oracle import fuzz_corrupt_port_vs_ref as fzc
    from oracle import fuzz_port_vs_ref as fz
    from test_oracle_golden import live_observations
    pre = WriteBatch().put(b"pre", b"x").data()
    corrupt = {}
    for seed in range(0, 25):
        mop, cs = fzc.cases(seed)
        corrupt[str(seed)] = []
        for bt, ts in cs:
            db = okv.Okv(ref, merge_op=mop)
            corrupt[str(seed)].append(fzc.recorded_outcome(fzc.outcome(db, pre, bt, ts)))
            db.close()
    tmp = tempfile.mkdtemp()
    try:
        return {"live": [digest(o) for o in live_observations(ref, ref_side=True)],
                "fuzz": {str(s): [digest(o) for o in fz.observe(s, ref)] for s in range(200, 212)},
                "corrupt_fuzz": corrupt,
                "sst_ingest": gen_sst_ingest(ref, tmp),
                "ingest_gpu": gen_ingest_gpu(ref, tmp)}
    finally:
        shutil.rmtree(tmp)


def main():
    if not okv.ref_available():
        raise SystemExit("oracle/_ref not built: run `make -C oracle ref` with the reference's sources at REF")
    ref = okv.load_ref()
    _sst_api(ref)
    os.makedirs(OUT, exist_ok=True)
    gen_ref_written(ref)
    for name, data in (("streams.json", gen_streams(ref)), ("corrupt.json", gen_corrupt(ref)),
                       ("known_answers.json", gen_known_answers(ref)), ("differential.json", gen_differential(ref))):
        with open(os.path.join(OUT, name), "w") as f:
            json.dump({"generator": "oracle/gen_golden.py", "source": "rocksdb_admin/tests/librocksdb.so.5.4",
                       "cases": data}, f, separators=(",", ":"))
        print(name, os.path.getsize(os.path.join(OUT, name)), "bytes")


if __name__ == "__main__":
    main()
