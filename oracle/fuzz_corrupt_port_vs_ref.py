"""Differential fuzzer for malformed WriteBatches: random mutations (byte flips, truncation, garbage tails, count and
tag edits) of valid batches through the oracle port and the reference's RocksDB — return code, error text, sequence
number, the latch on the next write, and the resulting contents must agree.  Test infrastructure only.
`python oracle/fuzz_corrupt_port_vs_ref.py FIRST LAST`."""
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import okv  # noqa: E402
from streams import random_stream  # noqa: E402


def mutate(rng, bt):
    b = bytearray(bt)
    r = rng.random()
    if r < 0.25 and len(b) > 0:
        for _ in range(rng.randint(1, 3)):
            b[rng.randrange(len(b))] = rng.getrandbits(8)
    elif r < 0.45:
        b = b[:rng.randrange(len(b) + 1)]
    elif r < 0.6:
        b += bytes(rng.getrandbits(8) for _ in range(rng.randint(1, 12)))
    elif r < 0.75 and len(b) >= 12:
        b[8:12] = (rng.choice([0, 1, 2, 255, 2 ** 32 - 1]) if rng.random() < 0.5 else rng.getrandbits(32)).to_bytes(4, "little")
    elif len(b) > 12:
        b[rng.randrange(12, len(b))] = rng.choice([0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 0x80, 0xff])
    return bytes(b)


def cases(seed, n=40):
    rng = random.Random(seed)
    mname = rng.choice(["counter", None, "append"])
    _, stream = random_stream(4000 + seed, n, n_keys=8, merge=mname, max_ops=rng.choice([1, 3, 6]))
    mop = {"counter": okv.MERGE_UINT64ADD, None: okv.MERGE_NONE, "append": okv.MERGE_APPEND}[mname]
    return mop, [(mutate(rng, bt), ts) for bt, ts in stream]


def outcome(db, pre, bt, ts):
    out = [db.apply(pre, 1)]
    out += [db.apply(bt, ts), db.last_error, db.latest_seq()]
    out += [db.apply(pre, 2), db.latest_seq()]  # the latch
    out.append(db.scan())
    return out


def recorded_outcome(o):
    """What tests/golden/differential.json keeps of the reference's outcome of one case: its return code and a digest"""
    from golden_util import digest
    return [o[1], digest(o)]


def run(first, last, a_lib=None, b_lib=None, make_a=None, recorded=None):
    """`recorded` ({seed: [recorded_outcome, ...]}) stands in for a live b_lib: the reference's outcomes stored by
    oracle/gen_golden.py, so the comparison runs where the reference's binary is not available."""
    from rocksplicator_b200.write_batch import WriteBatch
    pre = WriteBatch().put(b"pre", b"x").data()
    a_lib = a_lib or okv.load_port()
    if recorded is None:
        b_lib = b_lib or okv.load_ref()
    bad = known = 0
    for seed in range(first, last):
        mop, cs = cases(seed)
        for i, (bt, ts) in enumerate(cs):
            a = make_a(mop) if make_a else okv.Okv(a_lib, merge_op=mop)
            ra = outcome(a, pre, bt, ts)
            if recorded is None:
                b = okv.Okv(b_lib, merge_op=mop)
                rb = outcome(b, pre, bt, ts)
                b.close()
                same, b_rc, diff = ra == rb, rb[1], [x for x in zip(ra, rb) if x[0] != x[1]][:2]
            else:
                b_rc, b_digest = recorded[str(seed)][i]
                same, diff = recorded_outcome(ra) == [b_rc, b_digest], (ra[1:4], "reference rc", b_rc)
            if not same and ra[1] == 3 and b_rc == 0 and "outside the replicated hot path" in ra[2]:
                known += 1  # a well-formed range deletion: refused here, applied by RocksDB (DESIGN.md section 9)
            elif not same:
                bad += 1
                print("DIVERGE seed", seed, "case", i, bt.hex()[:120], diff)
            a.close()
    if known:
        print("known deviation (well-formed DeleteRange refused):", known)
    return bad


if __name__ == "__main__":
    print("done bad=", run(int(sys.argv[1]), int(sys.argv[2])))
