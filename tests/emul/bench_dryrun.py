"""TEST INFRASTRUCTURE — bench.py's whole control flow (load, compaction, MultiGet device + e2e, zipf, scans, apply
device + e2e, the mixed phase, the full-size parity assertions, the JSON line) on the CPU emulation at toy size, so that
an edit to bench.py or an API drift is caught without a GPU.  torch.cuda is replaced by no-op stand-ins (emulated
"device" pointers are host pointers, so CPU tensors serve as device buffers); timings are meaningless and ignored.

    python tests/emul/bench_dryrun.py [bench.py arguments]   # prints the JSON line bench.py would print
"""
import contextlib
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

from rocksplicator_b200 import engine  # noqa: E402


class _Event:
    def __init__(self, enable_timing=False):
        self.t = 0.0

    def record(self, stream=None):
        self.t = time.perf_counter()

    def synchronize(self):
        pass

    def elapsed_time(self, other):
        return max((other.t - self.t) * 1e3, 1e-3)


class _Stream:
    def __init__(self, stream_ptr=0, device=None, **kw):
        self.cuda_stream = int(stream_ptr or 0)

    def synchronize(self):
        pass

    def wait_stream(self, other):
        pass

    def wait_event(self, ev):
        pass


def _strip_device(fn):
    def wrapped(*a, **kw):
        if "device" in kw:
            kw = dict(kw)
            kw.pop("device")
        return fn(*a, **kw)
    return wrapped


def install():
    engine.SO_PATH = os.environ.get("RSP_TEST_EMUL_LIB", os.path.join(ROOT, "tests", "emul", "build", "librsp_b200_emul.so"))
    os.environ.setdefault("RSP_TEST_EMUL_HOST_LIB", os.path.join(os.path.dirname(engine.SO_PATH), "librsp_host_emul.so"))
    tc = torch.cuda
    tc.is_available = lambda: True
    tc.set_device = lambda *a, **k: None
    tc.synchronize = lambda *a, **k: None
    tc.Event = _Event
    tc.Stream = lambda *a, **k: _Stream(0)
    tc.ExternalStream = lambda ptr, device=None: _Stream(ptr)
    tc.stream = lambda s: contextlib.nullcontext()
    tc.current_stream = lambda *a, **k: _Stream(0)
    torch.Tensor.cuda = lambda self, *a, **k: self
    torch.Tensor.pin_memory = lambda self, *a, **k: self
    for name in ("empty", "zeros", "ones", "tensor", "full", "arange"):
        setattr(torch, name, _strip_device(getattr(torch, name)))
    torch.device = lambda *a, **k: "cpu"


def main(argv=None):
    install()
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    # arguments given here come after the toy-size defaults, so they add to them or override them
    sys.argv = ["bench.py", "--shards", "8", "--kv", "6000", "--mg-batches", "1", "--tick", "5", "--steps", "2",
                "--warmup", "1", "--no-cpu", "--big-tick", "40", "--c5-secs", "0.5"] + (argv or [])
    bench.main()


if __name__ == "__main__":
    main(sys.argv[1:])
