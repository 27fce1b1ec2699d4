"""Differential fuzzer: the oracle port (kv_oracle.c) against the reference's own RocksDB (oracle/_ref) on random
streams with flushes, compactions, MultiGets and iterator walks (Seek / SeekToFirst / SeekToLast / Next / Prev) at
random points.  Test infrastructure only.  `python oracle/fuzz_port_vs_ref.py FIRST_SEED LAST_SEED`; a short range
runs in tests/test_oracle_golden.py.  150 seeds: no divergence."""
import sys, random
import os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
from oracle import okv
from streams import random_stream
def iter_walk(db, keys, rng_seed):
    rng=random.Random(rng_seed)
    it=db.iterator(); out=[]
    for _ in range(30):
        r=rng.random()
        if r<0.2: it.seek_to_first(); out.append('F')
        elif r<0.4: it.seek_to_last(); out.append('L')
        elif r<0.6:
            k=rng.choice(keys); it.seek(k); out.append(('S',k))
        elif r<0.8:
            if it.valid(): it.next(); out.append('N')
        else:
            if it.valid(): it.prev(); out.append('P')
        out.append((it.valid(), it.key() if it.valid() else None, it.value() if it.valid() else None, it.status()))
    it.close()
    return out
def observe(seed, lib):
  """Everything one seed's run shows of `lib`, in order: (step, rc, error text) per batch, and (step, seq, MultiGet,
  iterator walk) at the random check points, then the final state.  The random choices do not depend on the results,
  so two libraries see the same calls."""
  rng=random.Random(seed*7+1)
  mop,mname=rng.choice([(okv.MERGE_COUNTER,"counter"),(okv.MERGE_APPEND,"append"),(okv.MERGE_UINT64ADD,"counter"),(okv.MERGE_NONE,None)])
  badops = (mop==okv.MERGE_COUNTER and rng.random()<0.3)
  keys,stream=random_stream(1000+seed, rng.randint(5,120), n_keys=rng.choice([3,10,40]), merge=mname, max_ops=rng.choice([2,6,20]), bad_operands=badops)
  db=okv.Okv(lib,merge_op=mop)
  out=[]
  for i,(bt,ts) in enumerate(stream):
      out.append((i, db.apply(bt,ts), db.last_error))
      if not badops and rng.random()<0.05:
          db.flush() if rng.random()<0.7 else db.compact()
      if rng.random()<0.1:
          out.append((i, db.latest_seq(), db.multi_get(keys), iter_walk(db,keys,i)))
  out.append(('end', db.latest_seq(), db.multi_get(keys), db.scan(), iter_walk(db,keys,99)))
  db.close()
  return out
def run(first, last, port=None, ref=None):
  port = port or okv.load_port(); ref = ref or okv.load_ref()
  bad = 0
  for seed in range(first, last):
      a=observe(seed, port); b=observe(seed, ref)
      if a!=b:
          i=next((j for j,(x,y) in enumerate(zip(a,b)) if x!=y), min(len(a),len(b)))
          bad+=1; print("DIVERGE", str((seed, i, a[i:i+1], b[i:i+1]))[:600])
  return bad


if __name__ == '__main__':
    print('done bad=', run(int(sys.argv[1]), int(sys.argv[2])))
