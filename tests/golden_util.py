"""Replay helpers shared by the oracle tests and the GPU parity tests.

A "db" is anything with the Okv method set: apply(batch, ts) -> rc, latest_seq(), get(k) -> (rc, v),
multi_get(keys) -> [(rc, v)], scan(start=None, limit=None), iterator() (seek/seek_to_last/next/prev/
valid/key/value/status/close), flush(), compact(), last_error.
"""
import hashlib
import json
import os

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MERGE_IDS = {"none": 0, "counter": 1, "uint64add": 2, "append": 3}


def load(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)["cases"]


def unhex(x):
    return None if x is None else bytes.fromhex(x)


def digest(obj):
    """Short stable fingerprint of an observation (nested tuples / lists of bytes, str, int, bool, None): lets the
    golden files hold what the reference returned for large results without storing the results themselves."""
    return hashlib.sha256(repr(obj).encode()).hexdigest()[:16]


def sha256(data):
    return hashlib.sha256(data).hexdigest()


def check_snapshot(db, keys, snap, tag=""):
    probe = list(keys) + [b"zz-missing"] + list(keys[:3])
    assert db.latest_seq() == snap["seq"], tag
    for (khex, rc, vhex), k in zip(snap["get"], probe):
        assert bytes.fromhex(khex) == k
        got = db.get(k)
        assert got == (rc, unhex(vhex)), (tag, "get", khex, got, rc, vhex)
    got = db.multi_get(probe)
    want = [(rc, unhex(v)) for rc, v in snap["multi_get"]]
    assert got == want, (tag, "multi_get")
    want_scan = [(bytes.fromhex(k), bytes.fromhex(v)) for k, v in snap["scan"]]
    assert db.scan() == want_scan, (tag, "scan")
    it = db.iterator()
    it.seek_to_last()
    rev = []
    while it.valid():
        rev.append((it.key(), it.value()))
        it.prev()
    assert rev == [(bytes.fromhex(k), bytes.fromhex(v)) for k, v in snap["rscan"]], (tag, "rscan")
    for khex, want in snap["seek"]:
        it.seek(bytes.fromhex(khex))
        if want is None:
            assert not it.valid(), (tag, "seek", khex)
        else:
            assert it.valid(), (tag, "seek", khex)
            assert (it.key(), it.value()) == (bytes.fromhex(want[0]), bytes.fromhex(want[1])), (tag, "seek", khex)
    assert it.status() == snap["iter_status"], (tag, "iter_status")
    it.close()


def replay_stream_case(db, case, flush_at=29, do_flush=True):
    keys = [bytes.fromhex(k) for k in case["keys"]]
    bad = case["name"] == "counter-2"  # malformed counter operands: the reference run did not flush
    for i, st in enumerate(case["steps"]):
        rc = db.apply(bytes.fromhex(st["batch"]), st["ts"])
        assert rc == st["rc"], (case["name"], i, rc, st["rc"], getattr(db, "last_error", ""))
        assert db.latest_seq() == st["seq"], (case["name"], i)
        if do_flush and i == flush_at and not bad:
            db.flush()
    if do_flush and not bad:
        db.compact()
    check_snapshot(db, keys, case["final"], case["name"])
