"""The engine's host logic and the kernels' LOGIC on a machine without a GPU: the engine's own sources compiled by g++
against tests/emul (a CPU emulation of the CUDA slice they use — threads as fibers, warp collectives, block barriers,
a malloc-backed runtime; TEST INFRASTRUCTURE, see tests/emul/include/cuda_runtime.h), and the `-m gpu` parity tests
re-run against that build in a subprocess.

What this is for: catching logic and addressing bugs before GPU time is spent (tests/emul/build_emul.py --asan runs
the same under AddressSanitizer).  What it is NOT: a product path, a fallback, or a parity claim — librsp_b200.so is
CUDA-only and the parity tests proper are the `-m gpu` runs on a B200.
"""
import importlib.util
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def emul():
    spec = importlib.util.spec_from_file_location("build_emul", os.path.join(ROOT, "tests", "emul", "build_emul.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build()


def _pytest_under_emulation(lib, extra_env, files, timeout=1500):
    env = dict(os.environ)
    env.update(extra_env)
    env["RSP_TEST_EMUL_LIB"] = lib
    env.setdefault("RSP_TEST_EMUL_ARENA", str(16 << 20))  # 16 MiB slabs: the emulated cudaMalloc poisons them (0xCD)
    p = subprocess.run([sys.executable, "-m", "pytest", "-m", "gpu", "-x", "-q", "-p", "no:cacheprovider"] + files,
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=timeout)
    print(p.stdout[-3000:], p.stderr[-2000:])
    assert p.returncode == 0, p.stdout[-3000:]
    return p.stdout


PARITY = ["tests/test_parity_gpu.py", "tests/test_zz_ingest_gpu.py"]


def test_parity_suite_under_emulation(emul):
    out = _pytest_under_emulation(emul[0], {}, PARITY)
    assert " passed" in out and "failed" not in out


def test_device_forms_under_emulation(emul):
    """tests/test_device_forms_gpu.py (the device-pointer entry points at every buffer shape, raw scan statuses, staged
    ticks) against the emulation"""
    out = _pytest_under_emulation(emul[0], {}, ["tests/test_device_forms_gpu.py"], timeout=900)
    assert " passed" in out and "failed" not in out


def test_compaction_runs_under_emulation(emul):
    """tests/test_compaction_gpu.py (every flushed and compacted run validated and compared with the host model of the
    merge rules) against the emulation"""
    out = _pytest_under_emulation(emul[0], {}, ["tests/test_compaction_gpu.py"], timeout=1500)
    assert " passed" in out and "failed" not in out


def test_router_over_two_emulated_devices(emul):
    """tests/test_router_gpu.py (two engines behind one router, maintenance on both) against the emulation"""
    out = _pytest_under_emulation(emul[0], {"RSP_EMUL_DEVICES": "2"}, ["tests/test_router_gpu.py"])
    assert "1 passed" in out


def test_engine_vs_oracle_fuzz_under_emulation(emul):
    """tests/emul/fuzz_engine_vs_port.py on a few dozen seeds (hundreds run in minutes from the command line)"""
    env = dict(os.environ)
    env.update({"RSP_TEST_EMUL_LIB": emul[0]})
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emul", "fuzz_engine_vs_port.py"), "3000", "3060"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    print(p.stdout[-2000:], p.stderr[-2000:])
    assert p.returncode == 0 and "done bad= 0" in p.stdout


def test_compaction_size_boundaries_under_emulation(emul):
    env = dict(os.environ)
    env.update({"RSP_TEST_EMUL_LIB": emul[0]})
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emul", "sweep_sizes.py")], cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=900)
    print(p.stdout[-1500:], p.stderr[-1500:])
    assert p.returncode == 0 and "SWEEP OK" in p.stdout


def test_engine_vs_oracle_corruption_fuzz_under_emulation(emul):
    """mutated WriteBatches: the decode kernel's error classes, texts, latch and all-or-nothing effect vs the oracle"""
    env = dict(os.environ)
    env.update({"RSP_TEST_EMUL_LIB": emul[0]})
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emul", "fuzz_corrupt_engine_vs_port.py"), "1000", "1030"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    print(p.stdout[-2000:], p.stderr[-2000:])
    assert p.returncode == 0 and "done bad= 0" in p.stdout


def test_bench_control_flow_under_emulation(emul, tmp_path):
    """bench.py end to end at toy size (tests/emul/bench_dryrun.py): every phase, its own full-size parity assertions
    and the JSON contract keys — an edit to bench.py or an API drift shows up here, not on the GPU box"""
    import json
    env = dict(os.environ)
    env["RSP_TEST_EMUL_LIB"] = emul[0]
    dump = tmp_path / "outputs"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emul", "bench_dryrun.py"), "--dump-outputs", str(dump)],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    print(p.stdout[-1500:], p.stderr[-2500:])
    assert p.returncode == 0
    line = json.loads(p.stdout.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"):
        assert key in line, key
    assert line["metric"] == "multiget_lookups_per_s"
    assert line["seams"]["ok"] and line["seams"]["applies_per_s"] > 0 and line["seams"]["multiget_lookups_per_s"] > 0
    assert set(line["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"}
    assert set(line["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"}
    assert "error" not in line["memtable"] and line["memtable"]["lookups_per_s"] > 0 and line["memtable"]["memtable_entries"] > 0
    assert "error" not in line["two_runs"] and line["two_runs"]["lookups_per_s"] > 0 and "2 sorted runs" in line["two_runs"]["what"]
    # --dump-outputs: the last timed step's results (bench_dryrun's toy size: 8 shards, 6000 KV, one MultiGet(4096) and
    # 8 x 5 batches per step, 1 warm-up + 2 timed steps), as float arrays
    import numpy as np
    from rocksplicator_b200 import synth
    out = {f.stem: np.load(f) for f in dump.glob("*.npy")}
    assert set(out) == {"multiget_lookup_index", "multiget_values", "multiget_value_len", "multiget_status", "apply_status"}
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert sum(f.stat().st_size for f in dump.glob("*.npy")) <= 64 << 20
    rng = np.random.default_rng(synth.SEED_QUERY)
    last = [rng.integers(0, 6000, size=4096, dtype=np.uint64) for _ in range(3)][-1]
    assert np.array_equal(out["multiget_lookup_index"], np.arange(4096))
    assert np.array_equal(out["multiget_values"], synth.values(synth.SEED_DATA, (last % np.uint64(8)).astype(np.int64), last, 0))
    assert (out["multiget_value_len"] == 64).all() and (out["multiget_status"] == 0).all()
    assert out["apply_status"].shape == (8 * 5,) and (out["apply_status"] == 0).all()


def test_host_mirror_over_emulated_engine(emul):
    """tests/cpp/host_tests.cpp's GpuDB-backed cases (replication chain, follower == leader, counter_service config 1,
    ApplicationDBManager, SST export / ingest) against the emulated engine"""
    for args in (["gpu-only"], ["gpu", "gpu_export_and_ingest"]):
        p = subprocess.run([emul[1]] + args, capture_output=True, text=True, timeout=900)
        print(p.stdout[-3000:], p.stderr[-1500:])
        assert p.returncode == 0 and " 0 failures" in p.stdout, p.stdout[-3000:]


def test_out_of_device_memory_paths(emul):
    """tests/emul/oom_probe.py with the emulated device capped at 8 MB: once the device is full applies are refused with an
    IO error (the flush that would make room cannot allocate), everything acknowledged before stays readable bit for bit,
    and applies go on after shards were closed.  (No GPU twin: driving a B200 out of memory under gpurun is a strike.)"""
    env = dict(os.environ)
    env.update({"RSP_TEST_EMUL_LIB": emul[0], "RSP_EMUL_DEVICE_BYTES": str(8 << 20)})
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emul", "oom_probe.py")], cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=900)
    print(p.stdout[-1500:], p.stderr[-1500:])
    assert p.returncode == 0 and "OOM PROBE OK" in p.stdout
