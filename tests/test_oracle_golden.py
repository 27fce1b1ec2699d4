"""Pins the oracle port (oracle/kv_oracle.c) to the reference:
  1. known-answer table measured on the reference's shipped librocksdb.so.5.4 (SURVEY.md §9),
  2. tests/golden/*.json generated from that binary by oracle/gen_golden.py,
  3. differential runs (random streams, fuzzers) against the binary's results for the same calls, recorded by
     oracle/gen_golden.py in tests/golden/differential.json.
CPU only.
"""
import struct

import pytest

import golden_util as G
from oracle import okv
from rocksplicator_b200.write_batch import WriteBatch
from streams import corrupt_cases, random_stream

u64 = lambda x: struct.pack("<Q", x)  # noqa: E731


def test_wire_format_sample():
    # SURVEY §9 "Wire format (confirmed byte-for-byte)" and §8 a6 probe sample
    b = WriteBatch().put(b"k1", b"v1").delete(b"k2").merge(b"c", u64(5)).put_log_data(u64(1234))
    assert b.data().hex() == ("0000000000000000" "03000000" "01026b31027631" "00026b32"
                              "020163080500000000000000" "0308d204000000000000")
    assert WriteBatch().put(b"key", b"value").data().hex() == "00000000000000000100000001036b65790576616c7565"
    assert WriteBatch().put(b"k" * 300, b"").data()[13:15] == bytes([0xAC, 0x02])


def test_port_known_answers(port_lib):
    """§9 rows 1-13/18 — the expectations are the committed outputs of the reference binary."""
    want = {r[0]: r[1:] for r in G.load("known_answers.json")}
    db = okv.Okv(port_lib, merge_op=okv.MERGE_UINT64ADD)
    assert [db.latest_seq()] == want["fresh_seq"]
    b = WriteBatch().put(b"k1", b"v1").delete(b"k2").merge(b"c", u64(5)).put_log_data(u64(1234)).set_sequence(999)
    assert [db.apply(b.data(), 5)] == want["row2_rc"]
    assert [db.latest_seq()] == want["row2_seq"] == [3]
    assert [db.apply(WriteBatch().put_log_data(u64(1)).data(), 5)] == want["row3_rc"]
    assert [db.latest_seq()] == want["row3_seq"]
    assert [db.apply(bytes(12), 5)] == want["row4_rc"]
    assert [db.latest_seq()] == want["row4_seq"]
    db.apply(WriteBatch().merge(b"c", u64(7)).data(), 5)
    assert [db.get(b"c")[1].hex()] == want["row5_get_c"]
    db.apply(WriteBatch().merge(b"k1", u64(1)).data(), 5)
    assert [db.get(b"k1")[1].hex()] == want["row6_get_k1"]
    db.apply(WriteBatch().put(b"z", u64(100)).delete(b"z").merge(b"z", u64(3)).merge(b"z", u64(4)).data(), 5)
    assert [db.latest_seq()] == want["row7_seq"]
    assert [db.get(b"z")[1].hex()] == want["row7_get_z"]
    db.apply(WriteBatch().put(b"x", b"1").put(b"x", b"2").delete(b"x").put(b"x", b"3").delete(b"y").data(), 5)
    assert [db.latest_seq()] == want["row8_seq"]
    assert [db.get(b"x")[1].hex()] == want["row8_get_x"]
    assert [db.get(b"y")[0]] == want["row8_get_y_rc"]
    db.apply(WriteBatch().put(b"", b"").put(b"ev", b"").data(), 5)
    assert [db.get(b"")[0], db.get(b"")[1].hex()] == want["row9_get_empty"]
    assert [[[k.hex(), v.hex()] for k, v in db.scan()]] == want["row10_scan"]
    assert [[[k.hex(), v.hex()] for k, v in db.scan(start=b"k", limit=1)]] == want["row10_seek_k"]
    mg = [[rc, v.hex() if v is not None else None] for rc, v in db.multi_get([b"c", b"zz", b"c", b"k2", b"ev", b""])]
    assert [mg] == want["row11_multi_get"]
    db.flush()
    assert [[[k.hex(), v.hex()] for k, v in db.scan()]] == want["row12_scan_after_flush"]
    assert [db.latest_seq()] == want["row12_seq"]
    db.apply(WriteBatch().single_delete(b"ev").data(), 5)
    assert [db.latest_seq()] == want["row18_seq"]
    assert [db.get(b"ev")[0]] == want["row18_get_ev_rc"]
    db.close()
    db = okv.Okv(port_lib, merge_op=okv.MERGE_NONE)
    assert [db.apply(WriteBatch().merge(b"m", b"1").data(), 5)] == want["row13_write_rc"]
    assert [db.latest_seq()] == want["row13_seq"]
    rc, _ = db.get(b"m")
    assert [rc, db.last_error] == want["row13_get_rc"]
    db.close()


@pytest.mark.parametrize("case", G.load("streams.json"), ids=lambda c: c["name"])
def test_port_golden_streams(port_lib, case):
    db = okv.Okv(port_lib, merge_op=G.MERGE_IDS[case["merge"]])
    G.replay_stream_case(db, case)
    db.close()


def test_port_golden_corrupt(port_lib):
    pre = WriteBatch().put(b"pre", b"x").data()
    for c in G.load("corrupt.json"):
        db = okv.Okv(port_lib, merge_op=okv.MERGE_UINT64ADD)
        assert db.apply(pre, 1) == 0
        assert db.apply(bytes.fromhex(c["batch"]), 0x1122334455667788) == c["rc"], c["name"]
        assert db.last_error == c["msg"], c["name"]
        assert db.latest_seq() == c["seq"], c["name"]
        assert db.apply(pre, 2) == c["rc_after"], c["name"]
        assert db.last_error == c["msg_after"], c["name"]
        assert db.latest_seq() == c["seq_after"], c["name"]
        assert [[k.hex(), v.hex()] for k, v in db.scan()] == c["scan"], c["name"]
        db.close()


def test_replicator_test_vectors(port_lib):
    """rocksdb_replicator/tests/rocksdb_replicator_test.cpp:146-208: 100 batches x 2 Puts -> follower seq
    200 and every key reads back; rocksdb_assumption_test.cpp:136-187: Put/Delete/Merge +1, batch of n +n."""
    db = okv.Okv(port_lib, merge_op=okv.MERGE_APPEND)
    for i in range(100):
        s = str(i).encode()
        wb = WriteBatch().put(s + b"key", s + b"value").put(s + b"key2", s + b"value2")
        assert db.apply(wb.data(), i) == 0
        assert db.latest_seq() == 2 * (i + 1)
    for i in range(100):
        s = str(i).encode()
        assert db.get(s + b"key") == (0, s + b"value")
        assert db.get(s + b"key2") == (0, s + b"value2")
    seq = db.latest_seq()
    db.apply(WriteBatch().delete(b"a").put(b"b", b"1").put(b"c", b"2").merge(b"b", b"3").data(), 0)
    assert db.latest_seq() == seq + 4
    assert db.get(b"b") == (0, b"13")
    db.close()


def live_observations(lib, ref_side):
    """The calls of test_port_vs_reference_live and what `lib` returns for each.  On the reference's side the stream
    is flushed after batch 40 and compacted at the end: the results must not depend on that."""
    out = []
    for mop, mname in ((okv.MERGE_COUNTER, "counter"), (okv.MERGE_APPEND, "append")):
        for seed in (91, 92):
            keys, stream = random_stream(seed + mop, 80, merge=mname)
            db = okv.Okv(lib, merge_op=mop)
            for i, (bt, ts) in enumerate(stream):
                out.append(db.apply(bt, ts))
                if ref_side and i == 40:
                    db.flush()
            if ref_side:
                db.compact()
            out.append((db.latest_seq(), [db.get(k) for k in keys], db.multi_get(keys), db.scan()))
            db.close()
    for name, bt in corrupt_cases():
        db = okv.Okv(lib, merge_op=okv.MERGE_UINT64ADD)
        out.append((name, db.apply(bt, 7), db.last_error, db.latest_seq()))
        db.close()
    return out


def test_port_vs_reference_live(port_lib):
    """Differential: random streams (not in the fixtures) through the port against the reference's results for the
    same calls (tests/golden/differential.json, recorded by oracle/gen_golden.py)."""
    want = G.load("differential.json")["live"]
    got = [G.digest(o) for o in live_observations(port_lib, ref_side=False)]
    assert len(got) == len(want)
    assert [i for i, (g, w) in enumerate(zip(got, want)) if g != w] == []


def _oracle_module(name):
    import importlib.util
    import os
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", name + ".py")
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_port_vs_reference_fuzz(port_lib):
    """oracle/fuzz_port_vs_ref.py on a few seeds: flush/compaction at random points, MultiGet, iterator walks; every
    observation against the reference's (tests/golden/differential.json)."""
    mod = _oracle_module("fuzz_port_vs_ref")
    want = G.load("differential.json")["fuzz"]
    assert sorted(want, key=int) == [str(s) for s in range(200, 212)]
    for seed in range(200, 212):
        got = [G.digest(o) for o in mod.observe(seed, port_lib)]
        assert got == want[str(seed)], seed


def test_port_vs_reference_corruption_fuzz(port_lib):
    """oracle/fuzz_corrupt_port_vs_ref.py on a few seeds: mutated batches, error class + text + latch + contents, against
    the reference's outcomes (tests/golden/differential.json)"""
    mod = _oracle_module("fuzz_corrupt_port_vs_ref")
    recorded = G.load("differential.json")["corrupt_fuzz"]
    assert sorted(recorded, key=int) == [str(s) for s in range(0, 25)]
    assert mod.run(0, 25, port_lib, recorded=recorded) == 0
