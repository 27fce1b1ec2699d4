"""Builds librsp_b200.so (CUDA kernels + engine + C ABI) in-tree with nvcc for sm_100a.

    python -m rocksplicator_b200.build [--force]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
import os
import subprocess
import sys
import tempfile
import zlib
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "librsp_b200.so")
SOURCES = ["k_apply.cu", "k_read.cu", "k_compact.cu", "engine.cu"]
HEADERS = ["format.cuh", "kernels.h", "stager.h", "arena.h", os.path.join("..", "..", "include", "rsp_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall"] + os.environ.get("RSP_NVCC_EXTRA", "").split()


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    jobs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + hdrs):
            jobs.append([_nvcc()] + NVCC_FLAGS + ["-c", s, "-o", o])

    def run(cmd):
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)

    with ThreadPoolExecutor(max_workers=4) as ex:
        list(ex.map(run, jobs))
    objs = [os.path.join(objdir, s.replace(".cu", ".o")) for s in SOURCES]
    if force or jobs or _stale(OUT, objs):
        run([_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", OUT] + objs +
            ["-cudart", "static", "-lpthread", "-ldl", "-lrt"])
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))


HOST = os.path.join(HERE, "host")
HOST_SRCS = ["gpu_db.cpp", "rocksdb_replicator/rocksdb_replicator.cpp", "rocksdb_replicator/gpu_db_wrapper.cpp",
             "rocksdb_admin/application_db.cpp", "rocksdb_admin/application_db_manager.cpp", "sst/sst_c_api.cpp",
             "bench/seam_bench.cpp", "rocksdb_admin/message_ingestion.cpp"]
HOST_SO = os.path.join(HERE, "librsp_host.so")
HOST_TESTS = os.path.join(os.path.dirname(HERE), "tests", "cpp", "host_tests")


def build_host(force=False, verbose=False):
    """The C++ mirror of the reference interfaces (host/) -> librsp_host.so, and its test binary."""
    build(force=False, verbose=verbose)
    srcs = [os.path.join(HOST, s) for s in HOST_SRCS]
    deps = list(srcs)
    for dp, _, fs in os.walk(HOST):
        deps += [os.path.join(dp, f) for f in fs if f.endswith(".h")]
    cxx = os.environ.get("CXX", "g++")
    flags = ["-std=c++17", "-O2", "-g", "-fPIC", "-Wall", "-I", HOST, "-pthread"]

    def run(cmd):
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)

    deps.append(os.path.join(os.path.dirname(HERE), "include", "rsp_b200.h"))  # (gpu_db.h includes the C ABI)
    if force or _stale(HOST_SO, deps + [OUT]):
        run([cxx] + flags + ["-shared", "-o", HOST_SO] + srcs + ["-L", HERE, "-lrsp_b200", "-Wl,-rpath,$ORIGIN"])
    tsrc = os.path.join(os.path.dirname(HERE), "tests", "cpp", "host_tests.cpp")
    tdeps = [tsrc, HOST_SO] + deps
    exe = HOST_TESTS
    if (force or _stale(exe, tdeps)) and not os.access(os.path.dirname(exe), os.W_OK):
        # the suite runs from a checkout whose tests/ is read-only: a test binary that has to be (re)linked goes to a
        # per-user directory outside the tree
        exe = os.path.join(tempfile.gettempdir(), "rsp_host_tests_%d_%08x" % (os.getuid(), zlib.crc32(HERE.encode())),
                           "host_tests")
        os.makedirs(os.path.dirname(exe), exist_ok=True)
    if force or _stale(exe, tdeps):
        run([cxx] + flags + ["-o", exe, tsrc, "-L", HERE, "-lrsp_host", "-lrsp_b200", "-Wl,-rpath," + HERE])
    return HOST_SO, exe
