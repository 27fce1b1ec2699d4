#!/usr/bin/env python
"""bench.py — the hot path of BASELINE.json on B200: MultiGet lookups/s + replicated applies/s per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]

Workload (BASELINE.json configs[1], SURVEY.md §8d "config 2"): 1024 shards on one GPU, 10 M KV total,
16 B keys / 64 B values, loaded through the apply path and fully compacted.  One step =
  * one MultiGet pass: 256 concurrent MultiGet(4096) calls = 1,048,576 uniform lookups in one launch, and
  * one apply tick: 1024 shards x 50 replicated single-Put WriteBatches (pull-sized, 105 wire bytes each).
`value` is MultiGet lookups/s with queries and results resident in HBM (CUDA events on the engine's
stream); `applies` carries the apply-side numbers; `e2e` is the same through the host-buffer C ABI
(rsp_multi_get_fixed / rsp_apply_many) with pinned host memory, H2D + D2H inside the timed region.
N > 1: one process per GPU (torchrun), each rank an independent engine with its own 1024 shards —
shards partition shard_id -> GPU, no collective on the data path ("scaling": "weak").
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

A_GET = 16 + (16 + 64 + 8) + 64          # algorithmic bytes per MultiGet hit (SURVEY §8d)
A_PUT = 83 + 22 + 88                     # per single-Put apply
DUMP_LOOKUPS = 65536                     # MultiGet results kept by --dump-outputs: 65536 x 64 values = 16 MB as float32


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def cpu_quota():
    """CPUs of time the container may use per second (cgroup v2 cpu.max / v1 cfs quota); None when uncapped.  The GPU
    boxes show 128 logical CPUs and cap the container at 16: every host-side figure is a figure under that quota."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        return None if q == "max" else float(q) / float(per)
    except Exception:
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else q / per
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def run_cpu(lib_kind, threads, shards, kv, apply_cap, get_secs, batch=4096, wal=1):
    """times oracle/okv_cpu_bench (the reference's RocksDB binary when build() left it in oracle/_ref, else the port)"""
    from oracle import okv
    okv.build(ref=False)
    lib = okv.REF_SO if (lib_kind == "reference" and okv.ref_available()) else okv.PORT_SO
    base = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
    d = os.path.join(base, "okv_bench_%d" % os.getpid())
    subprocess.call(["rm", "-rf", d])
    os.makedirs(d)
    try:
        out = subprocess.check_output([os.path.join(ROOT, "oracle", "okv_cpu_bench"), lib, str(threads), str(shards),
                                       str(kv), "64", str(wal), str(apply_cap), str(get_secs), str(batch), "1", d],
                                      text=True)
    finally:
        subprocess.call(["rm", "-rf", d])
    return json.loads(out.strip().splitlines()[-1])


class SeamCfg(C.Structure):
    _fields_ = [("device", C.c_int32), ("shards", C.c_uint32), ("kv_total", C.c_uint64), ("value_len", C.c_uint32),
                ("executor_threads", C.c_uint32), ("updates_per_response", C.c_uint32), ("update_rounds", C.c_uint32),
                ("multiget_threads", C.c_uint32), ("multiget_batch", C.c_uint32), ("multiget_secs", C.c_double),
                ("get_threads", C.c_uint32), ("get_secs", C.c_double), ("seed", C.c_uint64),
                ("first_shard_id", C.c_uint32), ("steady_rounds", C.c_uint32)]


class SeamResult(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("load_s", "load_applies_per_s", "resp_p50_ms", "resp_p99_ms", "compact_s",
                                          "mget_lookups_per_s", "mget_p50_ms", "mget_p99_ms")] + \
               [("mget_calls", C.c_uint64)] + \
               [(n, C.c_double) for n in ("get_per_s", "get_p50_us", "get_p99_us", "mixed_applies_per_s",
                                          "mixed_lookups_per_s", "mixed_resp_p50_ms", "mixed_resp_p99_ms")] + \
               [(n, C.c_uint64) for n in ("applied_total", "parity_errors", "status_errors", "engine_launches")] + \
               [(n, C.c_double) for n in ("steady_applies_per_s", "steady_resp_p50_ms", "steady_resp_p99_ms")] + \
               [("trace_us", C.c_double * 6), ("apply_comb", C.c_double * 9), ("read_comb", C.c_double * 5), ("cpu_s", C.c_double * 4)]


def run_seams(device, shards, kv, rank, world, secs=2.0, value_len=64, update_rounds=20, updates_per_response=50,
              reads=True, shard_base=0, steady_rounds=200):
    """The hot path through the reference's own seams (rocksplicator_b200/host/bench/seam_bench.cpp): followers pull
    from a synthetic leader through RocksDBReplicator -> DbWrapper; readers call ApplicationDB::MultiGet(4096) / Get from
    many threads.  Host buffers, H2D + D2H inside; every value checked against the generator."""
    from rocksplicator_b200 import build
    host_so = os.environ.get("RSP_TEST_EMUL_HOST_LIB")  # tests/emul/bench_dryrun.py only (CPU emulation, no timings)
    if not host_so:
        build.build_host()
        host_so = build.HOST_SO
    lib = C.CDLL(host_so)
    lib.rsp_seam_bench.restype = C.c_int
    lib.rsp_seam_bench.argtypes = [C.POINTER(SeamCfg), C.POINTER(SeamResult)]
    cores = os.cpu_count() or 8
    share = max(1, cores // max(1, world))
    cfg = SeamCfg(device=device, shards=shards, kv_total=kv, value_len=value_len,
                  executor_threads=max(16, min(32, share // 2)), updates_per_response=updates_per_response,
                  update_rounds=update_rounds if reads else 0,
                  multiget_threads=max(4, min(64, share // 2)) if reads else 0, multiget_batch=4096, multiget_secs=secs,
                  get_threads=max(8, min(256, share * 2)) if reads else 0, get_secs=secs / 2, seed=0x5EED0001 + rank,
                  first_shard_id=shard_base + rank * shards, steady_rounds=steady_rounds)
    res = SeamResult()
    rc = lib.rsp_seam_bench(C.byref(cfg), C.byref(res))
    out = {n: (list(getattr(res, n)) if n in ("trace_us", "apply_comb", "read_comb", "cpu_s") else getattr(res, n)) for n, _ in SeamResult._fields_}
    out["rc"] = rc
    out["threads"] = {"executor": cfg.executor_threads, "multiget": cfg.multiget_threads, "get": cfg.get_threads}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--kv", type=int, default=10_000_000)
    ap.add_argument("--shards", type=int, default=1024)
    ap.add_argument("--mg-batches", type=int, default=2048, help="concurrent MultiGet(4096) calls per launch")
    ap.add_argument("--tick", type=int, default=50, help="replicated updates per shard per apply tick")
    ap.add_argument("--cpu-kv", type=int, default=0, help="KV count of the CPU arm (0 = the same --kv as the GPU arm)")
    ap.add_argument("--big-tick", type=int, default=1000, help="updates per shard in the large apply tick (0 = skip)")
    ap.add_argument("--c5-secs", type=float, default=2.0, help="seconds of the config-5 sustained phase (0 = skip)")
    ap.add_argument("--cpu-get-secs", type=float, default=6.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-seams", action="store_true", help="skip the through-the-seams phase (librsp_host.so)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed step returned the last time as DIR/<name>.npy (float32 / float64, rank 0): "
                         "MultiGet values, lengths and statuses of a fixed sample of %d lookups, and the apply tick's "
                         "per-batch statuses; the same arguments give the same inputs" % DUMP_LOOKUPS)
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm returns no arrays")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    K, W = args.steps, max(args.warmup, 0)
    if not args.cpu_kv:
        args.cpu_kv = args.kv
    ncores = os.cpu_count() or 1
    workload = "%d shards x %d KV total, 16B key/64B value, uniform MultiGet batch=4096 x %d in flight, apply tick %d shards x %d single-Put WriteBatch" % (
        args.shards, args.kv, args.mg_batches, args.shards, args.tick)

    if args.impl == "reference":
        if rank != 0:
            return
        r = run_cpu("reference", ncores, args.shards, args.cpu_kv, 60.0, max(2.0, min(20.0, 1.0 * K)))
        line = {
            "impl": "reference", "metric": "multiget_lookups_per_s", "value": r["lookups_per_s"], "unit": "lookups/s",
            "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": 1e3 * r["get_s"] / max(K, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload, "sample": "%d KV applied (WAL on, default WriteOptions), flush+compact, %.0f s of MultiGet(4096) split per shard" % (r["applied"], r["get_s"])},
            "applies": {"value": r["applies_per_s"], "unit": "applies/s"},
            "cpu_baseline": {"value": r["lookups_per_s"], "unit": "lookups/s", "cores": r["threads"], "kind": r["kind"], "cpu_quota": cpu_quota(),
                             "sample": "%d KV over %d shards, %d threads" % (r["applied"], r["shards"], r["threads"]),
                             "applies_per_s": r["applies_per_s"]},
            "e2e": {"value": r["lookups_per_s"], "unit": "lookups/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    from rocksplicator_b200 import build, engine, synth
    if not os.path.exists(engine.SO_PATH):
        build.build()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # the timed regions run Python between engine calls: a generational collection over the setup's large object graph
    # inside ten timed ticks is a 70-80 ms stall (two of the r02 runs show exactly that in applies.e2e)
    import gc
    gc.collect()
    gc.freeze()
    gc.disable()
    lib = engine.load_library()
    eng = engine.Engine(local_rank, max_shards=max(16384, args.shards))
    stream = torch.cuda.ExternalStream(lib.rsp_engine_stream(eng.h), device=torch.device("cuda", local_rank))
    S, NKV = args.shards, args.kv
    shards = [eng.open_shard("segment%05d" % (rank * S + i), write_buffer_bytes=2 << 20) for i in range(S)]
    six_of = np.array([s.index for s in shards], dtype=np.uint32)
    seed = synth.SEED_DATA + rank

    # ---- load through the apply path, then fully compact -------------------------------------------
    t_load = time.perf_counter()
    CH = 1 << 20
    for lo in range(0, NKV, CH):
        idx = np.arange(lo, min(NKV, lo + CH), dtype=np.uint64)
        sh = (idx % np.uint64(S)).astype(np.int64)
        b = synth.single_put_batches(synth.keys16(seed, idx), synth.values(seed, sh, idx, 0), 1000 + idx)
        off = (np.arange(idx.size + 1, dtype=np.uint64) * np.uint64(b.shape[1]))
        st = eng.apply_packed(six_of[sh], b.reshape(-1), off, 1000 + idx)
        assert not st.any(), "load failed"
    eng.compact_all()
    t_load = time.perf_counter() - t_load
    assert sum(s.latest_seq() for s in shards) == NKV

    # ---- MultiGet: device-resident queries -----------------------------------------------------------
    Q = args.mg_batches * 4096
    n_sets = W + K
    rng = np.random.default_rng(synth.SEED_QUERY + rank)
    with torch.cuda.stream(stream):
        q_idx = [rng.integers(0, NKV, size=Q, dtype=np.uint64) for _ in range(n_sets)]
        d_keys = [torch.from_numpy(synth.keys16(seed, qi).reshape(-1)).cuda() for qi in q_idx]
        d_six = [torch.from_numpy(six_of[(qi % np.uint64(S)).astype(np.int64)].astype(np.int32)).cuda() for qi in q_idx]
        d_vals = torch.empty(Q * 64, dtype=torch.uint8, device="cuda")
        d_vlen = torch.empty(Q, dtype=torch.int32, device="cuda")
        d_st = torch.empty(Q, dtype=torch.int32, device="cuda")
    sp = C.c_void_p(stream.cuda_stream)

    def mg(i):
        rc = lib.rsp_multi_get_device(eng.h, Q, d_six[i].data_ptr(), d_keys[i].data_ptr(), 16, d_vals.data_ptr(), 64,
                                      d_vlen.data_ptr(), d_st.data_ptr(), sp)
        assert rc == 0

    for i in range(W):
        mg(i)
    barrier()
    clocks = ClockSampler(local_rank)
    clocks.start()
    launches0 = eng.kernel_launches()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    e_start, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_start.record(stream)
    for k in range(K):
        ev[k][0].record(stream)
        mg(W + k)
        ev[k][1].record(stream)
    e_end.record(stream)
    barrier()
    mg_total_ms = max_over_ranks(e_start.elapsed_time(e_end))
    mg_kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    mg_launches = eng.kernel_launches() - launches0
    # parity at full size (size-independent property: every value is a pure function of its key)
    last = q_idx[W + K - 1] if K else q_idx[-1]
    assert int(d_st.count_nonzero().item()) == 0 and int((d_vlen != 64).count_nonzero().item()) == 0
    want = synth.values(seed, (last % np.uint64(S)).astype(np.int64), last, 0)
    got = d_vals.cpu().numpy().reshape(Q, 64)
    assert np.array_equal(got, want), "MultiGet parity failed at full size"
    dump = {}
    if args.dump_outputs:  # the later phases reuse these buffers: sample them now
        rows = np.sort(np.random.default_rng(0).choice(Q, size=min(Q, DUMP_LOOKUPS), replace=False))
        dump["multiget_lookup_index"] = rows.astype(np.float64)
        dump["multiget_values"] = got[rows].astype(np.float32)
        dump["multiget_value_len"] = d_vlen.cpu().numpy()[rows].astype(np.float32)
        dump["multiget_status"] = d_st.cpu().numpy()[rows].astype(np.float32)

    # ---- config-2 variant: 10 % of the lookups ask for keys that were never written (NotFound) ------------
    with torch.cuda.stream(stream):
        m_idx = [rng.integers(0, NKV + NKV // 9, size=Q, dtype=np.uint64) for _ in range(3)]  # index >= NKV: absent
        m_keys = [torch.from_numpy(synth.keys16(seed, mi).reshape(-1)).cuda() for mi in m_idx]
        m_six = [torch.from_numpy(six_of[(mi % np.uint64(S)).astype(np.int64)].astype(np.int32)).cuda() for mi in m_idx]

    def mgm(i):
        j = i % 3
        assert lib.rsp_multi_get_device(eng.h, Q, m_six[j].data_ptr(), m_keys[j].data_ptr(), 16, d_vals.data_ptr(), 64,
                                        d_vlen.data_ptr(), d_st.data_ptr(), sp) == 0

    for i in range(W):
        mgm(i)
    barrier()
    ms0, ms1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms0.record(stream)
    for k in range(K):
        mgm(W + k)
    ms1.record(stream)
    barrier()
    miss_ms = max_over_ranks(ms0.elapsed_time(ms1))
    jm = (W + K - 1) % 3
    st_m = d_st.cpu().numpy()
    absent = m_idx[jm] >= np.uint64(NKV)
    assert np.array_equal(st_m != 0, absent) and (st_m[absent] == 1).all(), "miss variant: status"
    got_m0 = d_vals.cpu().numpy().reshape(Q, 64)[~absent]
    assert np.array_equal(got_m0, synth.values(seed, (m_idx[jm][~absent] % np.uint64(S)).astype(np.int64), m_idx[jm][~absent], 0)), "miss variant: values"
    miss_frac = float(absent.mean())
    # algorithmic bytes: a hit moves A_GET, a miss its key and status (SURVEY 8d: k + 8)
    a_miss_mix = (1.0 - miss_frac) * A_GET + miss_frac * (16 + 8)
    del m_keys, m_six

    # ---- zipf(0.99) MultiGet (config-4 access pattern on one GPU): hot keys are served from L2 ---------
    zrng = np.random.default_rng(synth.SEED_ZIPF + rank)
    z_idx = [synth.scatter_ranks(synth.zipf_ranks(zrng, NKV, 0.99, Q), NKV) for _ in range(3)]
    with torch.cuda.stream(stream):
        z_keys = [torch.from_numpy(synth.keys16(seed, zi).reshape(-1)).cuda() for zi in z_idx]
        z_six = [torch.from_numpy(six_of[(zi % np.uint64(S)).astype(np.int64)].astype(np.int32)).cuda() for zi in z_idx]

    def mgz(i):
        j = i % 3
        assert lib.rsp_multi_get_device(eng.h, Q, z_six[j].data_ptr(), z_keys[j].data_ptr(), 16, d_vals.data_ptr(), 64,
                                        d_vlen.data_ptr(), d_st.data_ptr(), sp) == 0

    for i in range(W):
        mgz(i)
    barrier()
    z0, z1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    z0.record(stream)
    for k in range(K):
        mgz(W + k)
    z1.record(stream)
    barrier()
    zipf_ms = max_over_ranks(z0.elapsed_time(z1))
    jz = (W + K - 1) % 3
    assert int(d_st.count_nonzero().item()) == 0
    assert np.array_equal(d_vals.cpu().numpy().reshape(Q, 64),
                          synth.values(seed, (z_idx[jz] % np.uint64(S)).astype(np.int64), z_idx[jz], 0)), "zipf MultiGet parity"

    # ---- MultiGet end to end: host (pinned) buffers through rsp_multi_get_fixed ------------------------
    h_keys = [torch.from_numpy(synth.keys16(seed, qi).reshape(-1)).pin_memory() for qi in q_idx[:min(n_sets, 4)]]
    h_six = [torch.from_numpy(six_of[(qi % np.uint64(S)).astype(np.int64)].astype(np.int32)).pin_memory() for qi in q_idx[:min(n_sets, 4)]]
    h_vals = torch.empty(Q * 64, dtype=torch.uint8).pin_memory()
    h_vlen = torch.empty(Q, dtype=torch.int32).pin_memory()
    h_st = torch.empty(Q, dtype=torch.int32).pin_memory()

    def mg_e2e(i):
        j = i % len(h_keys)
        rc = lib.rsp_multi_get_fixed(eng.h, Q, h_six[j].data_ptr(), h_keys[j].data_ptr(), 16, h_vals.data_ptr(), 64,
                                     h_vlen.data_ptr(), h_st.data_ptr())
        assert rc == 0

    for i in range(W):
        mg_e2e(i)
    barrier()
    t0 = time.perf_counter()
    for k in range(K):
        mg_e2e(W + k)
    barrier()
    mg_e2e_s = max_over_ranks(time.perf_counter() - t0)
    assert int(h_st.count_nonzero().item()) == 0
    jl = (W + K - 1) % len(h_keys)
    assert np.array_equal(h_vals.numpy().reshape(Q, 64),
                          synth.values(seed, (q_idx[jl] % np.uint64(S)).astype(np.int64), q_idx[jl], 0))

    # ---- range scans: Seek(random existing key) + 128 x Next, device-resident (config-4 shape on one GPU) --
    NSC, LSC = 16384, 128
    REC = 8 + 16 + 64
    sc_idx = [rng.integers(0, NKV, size=NSC, dtype=np.uint64) for _ in range(n_sets)]
    with torch.cuda.stream(stream):
        d_sk = [torch.from_numpy(synth.keys16(seed, qi).reshape(-1)).cuda() for qi in sc_idx]
        d_ss = [torch.from_numpy(six_of[(qi % np.uint64(S)).astype(np.int64)].astype(np.int32)).cuda() for qi in sc_idx]
        d_sout = torch.empty(NSC * LSC * REC, dtype=torch.uint8, device="cuda")
        d_snout = torch.empty(NSC, dtype=torch.int32, device="cuda")
        d_sst = torch.empty(NSC, dtype=torch.int32, device="cuda")

    def scan(i):
        rc = lib.rsp_multi_scan_device(eng.h, NSC, d_ss[i].data_ptr(), d_sk[i].data_ptr(), 16, LSC, d_sout.data_ptr(),
                                       LSC * REC, d_snout.data_ptr(), d_sst.data_ptr(), sp)
        assert rc == 0

    for i in range(W):
        scan(i)
    barrier()
    s_start, s_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s_start.record(stream)
    for k in range(K):
        scan(W + k)
    s_end.record(stream)
    barrier()
    sc_total_ms = max_over_ranks(s_start.elapsed_time(s_end))
    assert int(d_sst.count_nonzero().item()) == 0
    # parity: scan i of the last set returns the next keys of its shard in order, each with its value
    last_sc = sc_idx[W + K - 1] if K else sc_idx[-1]
    n_out = d_snout.cpu().numpy()
    entries_last = int(n_out.sum())
    per = NKV // S
    for qn in (0, 1, NSC // 2, NSC - 1):
        i0 = int(last_sc[qn]); sh0 = i0 % S; j0 = i0 // S
        cnt = int(n_out[qn])
        n_in_shard = len(range(sh0, NKV, S))
        assert cnt == min(LSC, n_in_shard - j0), (cnt, j0, n_in_shard)
        want_idx = np.arange(j0, j0 + cnt, dtype=np.uint64) * np.uint64(S) + np.uint64(sh0)
        got = d_sout[qn * LSC * REC: qn * LSC * REC + cnt * REC].cpu().numpy().reshape(cnt, REC)
        assert np.array_equal(got[:, 8:24], synth.keys16(seed, want_idx)), "scan keys"
        assert np.array_equal(got[:, 24:], synth.values(seed, np.full(cnt, sh0), want_idx, 0)), "scan values"
        assert (got[:, 0] == 16).all() and (got[:, 4] == 64).all()

    # ---- apply: replicated single-Put updates to existing keys, pull-sized groups per shard -----------
    T = S * args.tick
    ticks = []
    upd_idx = []
    ver_of = np.zeros(NKV, dtype=np.int32)  # newest version of every key, in application order of the ticks
    for stp in range(n_sets * 2):
        # `tick` updates per shard: shard-local ordinals uniform, global index = shard + ordinal * S
        per = NKV // S
        ordn = rng.integers(0, per, size=T, dtype=np.uint64)
        sh = np.repeat(np.arange(S, dtype=np.uint64), args.tick)
        idx = sh + ordn * np.uint64(S)
        b = synth.single_put_batches(synth.keys16(seed, idx), synth.values(seed, sh.astype(np.int64), idx, stp + 1), 5000 + idx)
        ticks.append((six_of[sh.astype(np.int64)], b, (np.arange(T + 1, dtype=np.uint64) * np.uint64(b.shape[1])), 5000 + idx))
        upd_idx.append(idx)
    staged = []
    for stp in range(n_sets):
        six, b, off, ts = ticks[stp]
        h = C.c_void_p()
        rc = lib.rsp_stage_build(eng.h, T, six.ctypes.data, b.ctypes.data, off.ctypes.data, ts.ctypes.data, C.byref(h))
        assert rc == 0
        staged.append(h)
    st_out = np.zeros(T, dtype=np.int32)

    def apply_dev(i):
        assert lib.rsp_reserve(eng.h, staged[i]) == 0
        assert lib.rsp_apply_staged_device(eng.h, staged[i], sp) == 0
        assert lib.rsp_apply_staged_finish(eng.h, staged[i], st_out.ctypes.data) == 0

    for i in range(W):
        apply_dev(i)
    barrier()
    launches1 = eng.kernel_launches()
    a_start, a_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # the K timed ticks go to the device back to back (each reserved against the ones still in flight); their
    # per-batch statuses are read back and folded into the host mirrors, in order, before the region ends
    bad_status = 0
    in_flight = []

    def fold():
        nonlocal bad_status
        for j in in_flight:
            assert lib.rsp_apply_staged_finish(eng.h, staged[j], st_out.ctypes.data) == 0
            bad_status += int(st_out.any())
        del in_flight[:]

    a_start.record(stream)
    for k in range(K):
        rc = lib.rsp_reserve(eng.h, staged[W + k])
        if rc == 11:  # Busy: a memtable is full while ticks are in flight — fold them, then it can be flushed
            fold()
            rc = lib.rsp_reserve(eng.h, staged[W + k])
        assert rc == 0
        assert lib.rsp_apply_staged_device(eng.h, staged[W + k], sp) == 0
        in_flight.append(W + k)
    fold()
    a_end.record(stream)
    assert bad_status == 0
    barrier()
    ap_total_ms = max_over_ranks(a_start.elapsed_time(a_end))
    ap_kernel_ms = eng.last_kernel_ms("apply")
    ap_launches = eng.kernel_launches() - launches1
    assert not st_out.any()
    if args.dump_outputs:  # fold() read the last tick's statuses last
        dump["apply_status"] = st_out.astype(np.float32)

    for stp in range(n_sets):
        ver_of[upd_idx[stp].astype(np.int64)] = stp + 1
    n_versions = 2 * n_sets + K  # version numbers used by the small ticks (device, e2e, mixed)

    # ---- the same with LARGE ticks (args.big_tick updates per shard): the bandwidth-bound regime of the tick -------
    big = None
    if args.big_tick:
        TB = S * args.big_tick
        KB, WB = min(K, 4), min(W, 2)
        per = NKV // S
        big_staged = []
        for stp in range(WB + KB):
            ordn = rng.integers(0, per, size=TB, dtype=np.uint64)
            shb = np.repeat(np.arange(S, dtype=np.uint64), args.big_tick)
            idxb = shb + ordn * np.uint64(S)
            vb = n_versions + 1 + stp
            bb = synth.single_put_batches(synth.keys16(seed, idxb), synth.values(seed, shb.astype(np.int64), idxb, vb), 7000 + idxb)
            sixb = six_of[shb.astype(np.int64)]
            offb = np.arange(TB + 1, dtype=np.uint64) * np.uint64(bb.shape[1])
            tsb = (7000 + idxb).astype(np.uint64)
            h = C.c_void_p()
            assert lib.rsp_stage_build(eng.h, TB, sixb.ctypes.data, bb.ctypes.data, offb.ctypes.data, tsb.ctypes.data, C.byref(h)) == 0
            big_staged.append(h)
            ver_of[idxb.astype(np.int64)] = vb
            del bb
        assert eng.flush_all() == 0  # empty memtables: the timed ticks fit without a flush in between
        stb = np.zeros(TB, dtype=np.int32)
        for i in range(WB):
            assert lib.rsp_reserve(eng.h, big_staged[i]) == 0
            assert lib.rsp_apply_staged_device(eng.h, big_staged[i], sp) == 0
            assert lib.rsp_apply_staged_finish(eng.h, big_staged[i], stb.ctypes.data) == 0 and not stb.any()
        barrier()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kern = []
        b0.record(stream)
        for k in range(KB):
            assert lib.rsp_reserve(eng.h, big_staged[WB + k]) == 0
            assert lib.rsp_apply_staged_device(eng.h, big_staged[WB + k], sp) == 0
            assert lib.rsp_apply_staged_finish(eng.h, big_staged[WB + k], stb.ctypes.data) == 0 and not stb.any()
            kern.append(eng.last_kernel_ms("apply"))
        b1.record(stream)
        barrier()
        big_ms = max_over_ranks(b0.elapsed_time(b1))
        big = {"batches_per_tick": TB, "ticks": KB, "ms_per_tick": big_ms / max(KB, 1), "kernel_ms_per_tick": float(np.mean(kern))}
        for h in big_staged:
            lib.rsp_stage_free(h)
        n_versions += WB + KB
    # back to one run per shard and empty memtables (untimed): the end-to-end ticks below then never meet a flush,
    # whose cost is what the config-5 phase measures
    assert eng.compact_all() == 0

    # e2e apply: pinned host buffers through rsp_apply_many (H2D + kernels + D2H of statuses inside)
    pinned_ticks = []
    for i in range(n_sets):
        six, b, off, ts = ticks[n_sets + i]
        pinned_ticks.append(tuple(torch.from_numpy(np.ascontiguousarray(x).reshape(-1)).pin_memory()
                                  for x in (six, b, off, ts.astype(np.uint64))))
    h_ast = torch.zeros(T, dtype=torch.int32).pin_memory()

    def apply_e2e(i):
        six_t, b_t, off_t, ts_t = pinned_ticks[i]
        rc = lib.rsp_apply_many(eng.h, T, six_t.data_ptr(), b_t.data_ptr(), off_t.data_ptr(), ts_t.data_ptr(),
                                h_ast.data_ptr())
        assert rc == 0 and int(h_ast.count_nonzero().item()) == 0

    for i in range(W):
        apply_e2e(i)
    barrier()
    t0 = time.perf_counter()
    e2e_tick_ms = []
    for k in range(K):
        tk = time.perf_counter()
        apply_e2e(W + k)
        e2e_tick_ms.append(1e3 * (time.perf_counter() - tk))
    barrier()
    ap_e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_tick_p50 = max_over_ranks(float(np.percentile(e2e_tick_ms, 50)))
    e2e_tick_p99 = max_over_ranks(float(np.percentile(e2e_tick_ms, 99)))
    clk = clocks.stop()
    for stp in range(n_sets, 2 * n_sets):
        ver_of[upd_idx[stp].astype(np.int64)] = stp + 1

    # ---- config 3: apply ticks and MultiGet launches CONCURRENTLY (two streams, lock-free memtable) --------
    mticks = []
    for stp in range(2 * n_sets, 2 * n_sets + K):
        per = NKV // S
        ordn = rng.integers(0, per, size=T, dtype=np.uint64)
        sh = np.repeat(np.arange(S, dtype=np.uint64), args.tick)
        idx = sh + ordn * np.uint64(S)
        b = synth.single_put_batches(synth.keys16(seed, idx), synth.values(seed, sh.astype(np.int64), idx, stp + 1), 5000 + idx)
        six = six_of[sh.astype(np.int64)]
        off = np.arange(T + 1, dtype=np.uint64) * np.uint64(b.shape[1])
        ts = 5000 + idx
        h = C.c_void_p()
        assert lib.rsp_stage_build(eng.h, T, six.ctypes.data, b.ctypes.data, off.ctypes.data, ts.ctypes.data, C.byref(h)) == 0
        mticks.append(h)
        upd_idx.append(idx)
    stream_b = torch.cuda.Stream(device=torch.device("cuda", local_rank))
    spb = C.c_void_p(stream_b.cuda_stream)
    barrier()
    mb0, mb1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ma0, ma1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stream_b.wait_stream(stream)
    t_mixed = time.perf_counter()
    mb0.record(stream_b)
    for k in range(K):  # reads: K launches queued on stream B
        assert lib.rsp_multi_get_device(eng.h, Q, d_six[W + k].data_ptr(), d_keys[W + k].data_ptr(), 16, d_vals.data_ptr(), 64,
                                        d_vlen.data_ptr(), d_st.data_ptr(), spb) == 0
    mb1.record(stream_b)
    ma0.record(stream)
    mixed_tick_ms = []
    for k in range(K):  # writes: K ticks on the engine stream while B runs
        tk = time.perf_counter()
        assert lib.rsp_reserve(eng.h, mticks[k]) == 0
        assert lib.rsp_apply_staged_device(eng.h, mticks[k], sp) == 0
        assert lib.rsp_apply_staged_finish(eng.h, mticks[k], st_out.ctypes.data) == 0
        mixed_tick_ms.append(1e3 * (time.perf_counter() - tk))  # launch -> statuses folded, the reads running beside it
        assert not st_out.any()
    ma1.record(stream)
    barrier()
    mixed_tick_p50 = max_over_ranks(float(np.percentile(mixed_tick_ms, 50))) if mixed_tick_ms else 0.0
    mixed_tick_p99 = max_over_ranks(float(np.percentile(mixed_tick_ms, 99))) if mixed_tick_ms else 0.0
    mixed_wall_s = max_over_ranks(time.perf_counter() - t_mixed)
    mixed_get_ms = max_over_ranks(mb0.elapsed_time(mb1))
    mixed_apply_ms = max_over_ranks(ma0.elapsed_time(ma1))
    # a lookup that raced a tick may see the value before or after it: every result is SOME version of its key
    assert int(d_st.count_nonzero().item()) == 0
    lastq = q_idx[W + K - 1] if K else q_idx[-1]
    samp = np.arange(0, Q, 64)
    got_m = d_vals.cpu().numpy().reshape(Q, 64)[samp]
    idx_m = lastq[samp]
    ok_m = np.zeros(samp.size, dtype=bool)
    for ver in range(0, n_versions + 1):
        todo = ~ok_m
        if not todo.any():
            break
        cand = synth.values(seed, (idx_m[todo] % np.uint64(S)).astype(np.int64), idx_m[todo], ver)
        ok_m[np.flatnonzero(todo)[(cand == got_m[todo]).all(axis=1)]] = True
    assert ok_m.all(), "mixed-phase MultiGet returned bytes that are no version of the key"
    for h in mticks:
        lib.rsp_stage_free(h)
    n_ticks_total = 2 * n_sets + K
    for stp in range(2 * n_sets, n_ticks_total):
        ver_of[upd_idx[stp].astype(np.int64)] = stp + 1

    # parity after the update ticks: the newest version wins for every updated key (last writer)
    chk = np.unique(np.concatenate([u[::97] for u in upd_idx]))
    ver = ver_of[chk.astype(np.int64)]
    res = eng.multi_get(six_of[(chk % np.uint64(S)).astype(np.int64)], [k.tobytes() for k in synth.keys16(seed, chk)], stride=64)
    for (rc, v), i, vr in zip(res, chk, ver):
        w = synth.values(seed, np.array([int(i) % S]), np.array([i], dtype=np.uint64), int(vr))[0].tobytes()
        assert rc == 0 and v == w, "apply parity failed"
    n_big_applied = (big["ticks"] + min(W, 2)) * big["batches_per_tick"] if big else 0
    assert sum(s.latest_seq() for s in shards) == NKV + n_ticks_total * T + n_big_applied

    # ---- config-2 variant: MultiGet while the newest version of many keys is still in the memtables -----
    # (every update tick above landed in a memtable: nothing has been flushed since the load).  Informational: a
    # failure here fails the bench (r01: informational).
    def mg_phase_checked():
        """W + K MultiGet launches of the uniform query sets, K of them timed; status, length and (full size) values
        checked against the last update tick of every queried key.  Local to the rank: no collectives inside."""
        for i in range(W):
            mg(i)
        torch.cuda.synchronize()
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        m0.record(stream)
        for k in range(K):
            mg(W + k)
        m1.record(stream)
        torch.cuda.synchronize()
        ms = float(m0.elapsed_time(m1))
        assert int(d_st.count_nonzero().item()) == 0 and int((d_vlen != 64).count_nonzero().item()) == 0, "status / length"
        lastq = q_idx[W + K - 1] if K else q_idx[-1]
        qver = ver_of[lastq.astype(np.int64)]
        got = d_vals.cpu().numpy().reshape(Q, 64)
        qsh = (lastq % np.uint64(S)).astype(np.int64)
        for v in np.unique(qver):
            m = qver == v
            assert np.array_equal(got[m], synth.values(seed, qsh[m], lastq[m], int(v))), "value parity (version %d)" % v
        return ms

    mt_err = None
    mt_entries = int(sum(s.stats()["memtable_entries"] for s in shards))
    mt_ms = mg_phase_checked()

    # ---- the same once more after a flush WITHOUT compaction: every shard now has two sorted runs (the state between a
    # flush and the merge at level0_file_num_compaction_trigger; config 5 lives there).
    r2_err = None
    assert eng.flush_all() == 0
    r2_runs = int(max(s.stats()["n_runs"] for s in shards))
    r2_ms = mg_phase_checked()

    # ---- config 5 shape on this GPU: 256-byte values, 80 % applies / 20 % lookups by operation count, flushes and
    # merges happening as the memtables fill (BASELINE configs[4]; options examples/counter_service/rocksdb_options.cpp:78-93)
    c5 = None
    if args.c5_secs > 0:
        V5, PER5 = 256, 2048
        N5 = S * PER5
        c5_shards = [eng.open_shard("cfive%05d" % (rank * S + i), write_buffer_bytes=2 << 20) for i in range(S)]
        c5_six = np.array([s.index for s in c5_shards], dtype=np.uint32)
        seed5 = seed + 0x500
        for lo in range(0, N5, 1 << 19):
            idx = np.arange(lo, min(N5, lo + (1 << 19)), dtype=np.uint64)
            sh = (idx % np.uint64(S)).astype(np.int64)
            b = synth.single_put_batches(synth.keys16(seed5, idx), synth.values(seed5, sh, idx, 0, V5), 9000 + idx)
            order = np.argsort(sh, kind="stable")
            off = np.arange(idx.size + 1, dtype=np.uint64) * np.uint64(b.shape[1])
            st = eng.apply_packed(c5_six[sh[order]], np.ascontiguousarray(b[order]).reshape(-1), off, (9000 + idx[order]))
            assert not st.any()
        stats0 = [s_.stats() for s_ in c5_shards]
        # a rotating set of pre-built ticks (80 % of the operations) and query sets (20 %)
        T5, Q5, NT5 = S * 50, S * 50 // 4, 8
        t5 = []
        ver5 = np.zeros(N5, dtype=np.int32)
        for i in range(NT5):
            ordn = rng.integers(0, PER5, size=T5, dtype=np.uint64)
            sh = np.repeat(np.arange(S, dtype=np.uint64), 50)
            idx = sh + ordn * np.uint64(S)
            b = synth.single_put_batches(synth.keys16(seed5, idx), synth.values(seed5, sh.astype(np.int64), idx, i + 1, V5), 9000 + idx)
            t5.append(tuple(torch.from_numpy(np.ascontiguousarray(x).reshape(-1)).pin_memory() for x in (
                c5_six[sh.astype(np.int64)], b, np.arange(T5 + 1, dtype=np.uint64) * np.uint64(b.shape[1]), (9000 + idx).astype(np.uint64))) + (idx.astype(np.int64),))
        q5 = [rng.integers(0, N5, size=Q5, dtype=np.uint64) for _ in range(NT5)]
        q5k = [torch.from_numpy(synth.keys16(seed5, q).reshape(-1)).pin_memory() for q in q5]
        q5s = [torch.from_numpy(c5_six[(q % np.uint64(S)).astype(np.int64)]).pin_memory() for q in q5]
        h5_vals = torch.empty(Q5 * V5, dtype=torch.uint8).pin_memory()
        h5_vlen = torch.empty(Q5, dtype=torch.int32).pin_memory()
        h5_st = torch.empty(Q5, dtype=torch.int32).pin_memory()
        h5_ast = torch.zeros(T5, dtype=torch.int32).pin_memory()
        barrier()
        n_ticks5 = 0
        compact_ms0 = max(0.0, eng.last_kernel_ms("compact_total"))
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < args.c5_secs:
            i = n_ticks5 % NT5
            six_t, b_t, off_t, ts_t, idx_t = t5[i]
            assert lib.rsp_apply_many(eng.h, T5, six_t.data_ptr(), b_t.data_ptr(), off_t.data_ptr(), ts_t.data_ptr(), h5_ast.data_ptr()) == 0
            ver5[idx_t] = i + 1
            assert lib.rsp_multi_get_fixed(eng.h, Q5, q5s[i].data_ptr(), q5k[i].data_ptr(), 16, h5_vals.data_ptr(), V5, h5_vlen.data_ptr(), h5_st.data_ptr()) == 0
            n_ticks5 += 1
        c5_s = time.perf_counter() - t0
        assert int(h5_ast.count_nonzero().item()) == 0 and int(h5_st.count_nonzero().item()) == 0
        il = (n_ticks5 - 1) % NT5
        assert np.array_equal(h5_vals.numpy().reshape(Q5, V5)[::7],
                              np.concatenate([synth.values(seed5, np.array([int(q) % S]), np.array([q], dtype=np.uint64), int(ver5[int(q)]), V5) for q in q5[il][::7]])), "config-5 lookup parity"
        stats1 = [s_.stats() for s_ in c5_shards]
        d = lambda k: sum(b_[k] - a_[k] for a_, b_ in zip(stats0, stats1))  # noqa: E731
        ingested = n_ticks5 * T5 * (16 + V5 + 8)  # bytes of entries written by the applies (k + v + 8 each)
        c5_local = {"ticks": n_ticks5, "secs": c5_s, "applies": n_ticks5 * T5, "lookups": n_ticks5 * Q5, "flushes": d("flushes"),
                    "compactions": d("compactions"), "bytes_read": d("compaction_bytes_read"), "bytes_written": d("compaction_bytes_written"),
                    "ingested": ingested, "max_runs": max(s_["n_runs"] for s_ in stats1), "compact_ms": max(0.0, eng.last_kernel_ms("compact_total")) - compact_ms0}
        c5 = {k: sum_over_ranks(float(v)) for k, v in c5_local.items() if k not in ("secs", "max_runs")}
        c5["secs"] = max_over_ranks(c5_local["secs"])
        c5["max_runs"] = max_over_ranks(float(c5_local["max_runs"]))
        for s_ in c5_shards:
            s_.close()

    # ---- numbers ---------------------------------------------------------------------------------------
    peak, peak_src = peaks()
    # every collective is issued by every rank, before any rank-0-only code
    tot_lookups = sum_over_ranks(Q * K)
    mt_ms_all = max_over_ranks(mt_ms)
    mt_failed = sum_over_ranks(1.0 if mt_err else 0.0)
    mt_entries_all = sum_over_ranks(float(mt_entries))
    r2_ms_all = max_over_ranks(r2_ms)
    r2_failed = sum_over_ranks(1.0 if r2_err else 0.0)
    tot_applies = sum_over_ranks(T * K)
    tot_scans = sum_over_ranks(NSC * K)
    tot_scan_entries = sum_over_ranks(entries_last * K)
    lookups_per_s = tot_lookups / (mg_total_ms * 1e-3)
    applies_per_s = tot_applies / (ap_total_ms * 1e-3)
    ach = A_GET * Q / (mg_kernel_ms * 1e-3) / 1e9
    # DRAM traffic of the roofline kernel cannot be measured inside a timed run: it is what one `ncu --set full` capture of
    # this same command recorded (dram__bytes_read.sum + dram__bytes_write.sum for one launch), kept under profiles/
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "multiget_traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            if tj.get("lookups_per_launch") == Q:
                traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
        except Exception:
            traffic = None
    # ---- the same path through the reference's seams: DbWrapper (pull loop) and ApplicationDB (MultiGet / Get) ------
    seams = None
    if not args.no_seams:
        for h in staged:
            lib.rsp_stage_free(h)
        staged = []
        barrier()
        try:
            seams = run_seams(local_rank, S, NKV, rank, world)
            # the pull protocol keeps ONE response in flight per shard (replicated_db.cpp:430): its size is the reference's
            # flag replicator_max_updates_per_response (default 50).  The same pull loops with 500 updates per response:
            big_resp = run_seams(local_rank, S, min(NKV, S * 4000), rank, world, updates_per_response=500, reads=False,
                                 shard_base=20000, steady_rounds=0)
            seams["load500_applies_per_s"] = big_resp.get("load_applies_per_s", 0.0) if big_resp.get("rc") == 0 and not big_resp.get("status_errors") else 0.0
            seams["load500_p50_ms"] = big_resp.get("resp_p50_ms", 0.0)
        except Exception as ex:  # noqa: BLE001
            seams = {"rc": -1, "error": "%s: %s" % (type(ex).__name__, str(ex)[:200])}
        ok = 1.0 if (seams.get("rc") == 0 and seams.get("parity_errors") == 0 and seams.get("status_errors") == 0) else 0.0
        seams_all_ok = sum_over_ranks(ok) == world
        seams_sum = {k: sum_over_ranks(float(seams.get(k, 0.0))) for k in (
            "load_applies_per_s", "mget_lookups_per_s", "get_per_s", "mixed_applies_per_s", "mixed_lookups_per_s", "load500_applies_per_s",
            "steady_applies_per_s")}
        seams_max = {k: max_over_ranks(float(seams.get(k, 0.0))) for k in (
            "resp_p50_ms", "resp_p99_ms", "mget_p50_ms", "mget_p99_ms", "get_p50_us", "get_p99_us", "mixed_resp_p50_ms",
            "mixed_resp_p99_ms", "steady_resp_p50_ms", "steady_resp_p99_ms")}
    cpu = None
    if rank == 0 and args.gpus == 1 and not args.no_cpu:
        r = run_cpu("reference", ncores, S, args.cpu_kv, 60.0, args.cpu_get_secs)
        cpu = {"value": r["lookups_per_s"], "unit": "lookups/s", "cores": r["threads"], "kind": r["kind"],
               "sample": "%d KV applied over %d shards with default WriteOptions (WAL on), flush+compact, then %.0f s of MultiGet(4096) split per shard; %d threads" % (
                   r["applied"], r["shards"], r["get_s"], r["threads"]),
               "applies_per_s": r["applies_per_s"],
               "cpu_quota": cpu_quota(),
               "per_core": {"lookups_per_s": r["lookups_per_s"] / max(1.0, min(r["threads"], cpu_quota() or r["threads"])),
                            "applies_per_s": r["applies_per_s"] / max(1.0, min(r["threads"], cpu_quota() or r["threads"])),
                            "what": "per CPU of time available: min(threads, the container's CPU quota)"},
               "note": "the reference's options share one LRU block cache per DB among all reader threads; per-core figures are the fair comparison"}
    # (collectives are issued by every rank: none inside the rank-0 block below)
    big_applies_all = sum_over_ranks(big["batches_per_tick"] * big["ticks"]) if big else 0.0
    if rank == 0:
        line = {
            "metric": "multiget_lookups_per_s", "value": lookups_per_s, "unit": "lookups/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": (mg_total_ms + ap_total_ms) / max(K, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload, "l2": "inputs larger than L2: %.2f GB entry heap per GPU, fresh uniform keys every step" % (NKV * 96 / 1e9),
                       "timing": "CUDA events on the engine stream, max over ranks", "load_s": round(t_load, 2),
                       "flags": {k: os.environ[k] for k in sorted(os.environ) if k.startswith("RSP_")}},
            "applies": {"value": applies_per_s, "unit": "applies/s", "ms_per_tick": ap_total_ms / max(K, 1),
                        "kernel_ms_last_tick": ap_kernel_ms, "batches_per_tick": T,
                        "what": "device-resident: the ticks are pre-staged device images (rsp_stage_build, H2D outside the timed region); the K ticks are launched back to back, statuses read back and folded, in order, inside the timed region",
                        "large_ticks": (None if not big else dict(big, applies_per_s=big_applies_all / (big["ms_per_tick"] * big["ticks"] * 1e-3),
                                                                  hbm_frac_of_peak=A_PUT * big["batches_per_tick"] / (big["kernel_ms_per_tick"] * 1e-3) / 1e9 / peak)),
                        "hbm_frac_of_peak": (A_PUT * T / (ap_kernel_ms * 1e-3) / 1e9 / peak) if ap_kernel_ms and ap_kernel_ms > 0 else None,
                        "e2e": {"value": tot_applies / ap_e2e_s, "unit": "applies/s", "h2d_bytes_per_step": int(ticks[0][1].size + 10 * T), "d2h_bytes_per_step": 4 * T + 24 * S,
                                "tick_ms": {"p50": e2e_tick_p50, "p99": e2e_tick_p99, "what": "one rsp_apply_many call of %d batches from pinned host memory, host clock" % T}}},
            "roofline": {"kernel": "k_multi_get16", "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes_per_lookup": A_GET,
                         "lookups_per_launch": Q, "launch_ms": mg_kernel_ms},
            "memtable": ({"error": mt_err or "failed on another rank"} if mt_failed else
                         {"what": "config-2 variant: the same uniform MultiGet with the update ticks still in the memtables (entries there = %.0f %% of the key count; nothing flushed since the load); values checked at full size" % (100.0 * mt_entries_all / max(1, NKV * world)),
                          "lookups_per_s": tot_lookups / (mt_ms_all * 1e-3), "memtable_entries": int(mt_entries_all),
                          "hbm_frac_of_peak_algorithmic": A_GET * Q / (mt_ms_all * 1e-3 / max(K, 1)) / 1e9 / peak}),
            "two_runs": ({"error": r2_err or "failed on another rank"} if r2_failed else
                         {"what": "the same MultiGet after a flush without compaction: %d sorted runs per shard (lookups that miss the newest run go on to the older one); values checked at full size" % r2_runs,
                          "lookups_per_s": tot_lookups / (r2_ms_all * 1e-3),
                          "hbm_frac_of_peak_algorithmic": A_GET * Q / (r2_ms_all * 1e-3 / max(K, 1)) / 1e9 / peak}),
            "miss10": {"what": "config-2 variant: %.1f %% of the lookups ask for keys that were never written (NotFound); statuses and the values of the hits checked at full size" % (100 * miss_frac),
                       "lookups_per_s": tot_lookups / (miss_ms * 1e-3),
                       "hbm_frac_of_peak_algorithmic": a_miss_mix * Q / (miss_ms * 1e-3 / max(K, 1)) / 1e9 / peak},
            "config5": (None if not c5 else {
                "what": "config-5 shape per GPU: %d shards, 16 B keys / 256 B values, alternating apply ticks (80 %% of the operations, %d single-Put WriteBatches each) and MultiGet calls (20 %%) through the host-buffer C ABI for %.1f s, flushes and size-tiered merges running as the memtables fill" % (S, S * 50, args.c5_secs),
                "applies_per_s": c5["applies"] / c5["secs"], "lookups_per_s": c5["lookups"] / c5["secs"],
                "flushes": int(c5["flushes"]), "merges": int(c5["compactions"]), "max_runs_per_shard": int(c5["max_runs"]),
                "write_amplification": c5["bytes_written"] / max(1.0, c5["ingested"]),
                "compaction": {"bytes_read": c5["bytes_read"], "bytes_written": c5["bytes_written"], "kernel_ms": c5["compact_ms"],
                               "hbm_frac_of_peak": ((c5["bytes_read"] + c5["bytes_written"]) / max(1e-9, c5["compact_ms"] * 1e-3 / max(1, world)) / 1e9 / peak) if c5["compact_ms"] > 0 else None}}),
            "zipf": {"theta": 0.99, "lookups_per_s": tot_lookups / (zipf_ms * 1e-3), "hbm_frac_of_peak_algorithmic": A_GET * Q / (zipf_ms * 1e-3 / max(K, 1)) / 1e9 / peak},
            "mixed": {"what": "config 3: %d apply ticks on the engine stream concurrent with %d MultiGet launches on a second stream" % (K, K),
                      "lookups_per_s": tot_lookups / (mixed_get_ms * 1e-3), "applies_per_s": tot_applies / (mixed_apply_ms * 1e-3),
                      "wall_ms": mixed_wall_s * 1e3,
                      "tick_ms": {"p50": mixed_tick_p50, "p99": mixed_tick_p99, "what": "one pre-staged tick: launch to statuses folded on the host (host clock)"}},
            "scans": {"value": tot_scans / (sc_total_ms * 1e-3), "unit": "scans/s", "entries_per_s": tot_scan_entries / (sc_total_ms * 1e-3),
                      "scan_len": LSC, "scans_per_launch": NSC,
                      "hbm_frac_of_peak": (entries_last * 168 + 16 * NSC) / (sc_total_ms * 1e-3 / max(K, 1)) / 1e9 / peak},
            "e2e": {"value": tot_lookups / mg_e2e_s, "unit": "lookups/s", "h2d_bytes_per_step": Q * 20, "d2h_bytes_per_step": Q * 72},
            "seams": (None if seams is None else {
                "what": "the same path through the reference's seams (librsp_host.so): %d follower pull loops (RocksDBReplicator -> DbWrapper::HandleReplicateResponses, 50 updates per response, synthetic leader behind the Transport interface) load %d KV; ApplicationDB::MultiGet(4096 keys of one shard) and ApplicationDB::Get from caller threads; host std::string / Slice buffers, H2D + D2H inside; values checked against the generator" % (S * world, NKV * world),
                "ok": bool(seams_all_ok), "threads_per_rank": seams.get("threads"), "error": seams.get("error"),
                "applies_per_s": seams_sum["load_applies_per_s"], "response_to_next_pull_ms": {"p50": seams_max["resp_p50_ms"], "p99": seams_max["resp_p99_ms"]},
                "steady": {"what": "the pull loops alone on the loaded shards (200 more responses per shard, flushes running as the memtables fill): the sustained follower rate",
                           "applies_per_s": seams_sum["steady_applies_per_s"],
                           "response_to_next_pull_ms": {"p50": seams_max["steady_resp_p50_ms"], "p99": seams_max["steady_resp_p99_ms"]},
                           "round_trip_stage_us_rank0": dict(zip(("transport", "to_executor", "handle_and_stage", "engine", "to_continuation", "to_next_pull"), seams.get("trace_us") or [])),
                           "apply_combiner_rank0": dict(zip(("batches", "updates", "ms_running", "ms_waiting_copiers", "ms_idle", "sum_ms_call_to_batch_ran", "sum_ms_to_callback_start", "sum_ms_in_callbacks", "callbacks"), seams.get("apply_comb") or []))},
                "get_combiner_rank0": dict(zip(("batches", "keys", "ms_running", "ms_waiting_copiers", "ms_idle"), seams.get("read_comb") or [])),
                "cpu_seconds_rank0": dict(zip(("load", "multiget", "get", "steady"), seams.get("cpu_s") or [])),
                "applies_per_s_at_500_updates_per_response": seams_sum["load500_applies_per_s"],
                "note": "one response in flight per shard (the pull protocol): applies/s = shards x updates per response / round trip; 50 per response is the reference's default flag, 500 shows the same loops with a larger flag value",
                "multiget_lookups_per_s": seams_sum["mget_lookups_per_s"], "multiget_call_ms": {"p50": seams_max["mget_p50_ms"], "p99": seams_max["mget_p99_ms"]},
                "get_per_s": seams_sum["get_per_s"], "get_call_us": {"p50": seams_max["get_p50_us"], "p99": seams_max["get_p99_us"]},
                "mixed": {"what": "config 3: replicated updates flowing through the pull loops while MultiGet runs",
                          "applies_per_s": seams_sum["mixed_applies_per_s"], "lookups_per_s": seams_sum["mixed_lookups_per_s"],
                          "response_to_next_pull_ms": {"p50": seams_max["mixed_resp_p50_ms"], "p99": seams_max["mixed_resp_p99_ms"]}},
                "rank0": {k: seams.get(k) for k in ("load_s", "compact_s", "mget_calls", "applied_total", "parity_errors", "status_errors", "engine_launches")}}),
            "cpu_baseline": cpu,
            "host": {"cpus_visible": ncores, "cpu_quota": cpu_quota(),
                     "note": "figures through host buffers / the seams are bounded by the container's CPU time"},
            "gpu_launches": int(mg_launches + ap_launches),
            "clocks": clk,
        }
        print(json.dumps(line))
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in dump.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    for h in staged:
        lib.rsp_stage_free(h)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
