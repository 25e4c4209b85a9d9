"""Dry run of ``bench.py``'s GPU arm on a box WITHOUT GPUs: the same function (``bench.run_b200_arm``), the same front
door (real ``modin.pandas`` + plug-in when oracle/_ref is installed), the same legs, checks and collectives -- on the
numpy device double (tests/cpu_double.py), under gloo, with ``torch.cuda.*`` replaced by host stand-ins and tiny frames.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29655 \
        tests/bench_dryrun.py --rows 400000

What it is for: the control flow of the bench at world sizes this container has no GPUs for -- that every rank reaches
every collective (a leg that only some ranks enter is a hang on the real box), that the JSON line is well formed and
that every ``checked`` / ``parity_ok`` is true.  It measures nothing.  Test infrastructure only
(tests/test_bench_dryrun.py runs it at world sizes 1, 2 and 8).
"""

import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402
import torch  # noqa: E402


class _Event:
    def __init__(self, enable_timing=True):
        self.t = None

    def record(self, stream=None):
        self.t = time.perf_counter()

    def elapsed_time(self, other):
        return max((other.t - self.t) * 1e3, 1e-6)


class _Stream:
    cuda_stream = 0

    def synchronize(self):
        pass


def main():
    os.environ["MB200_BENCH_DEVICE"] = "cpu"
    hang_after = float(os.environ.get("MB200_DRYRUN_HANG_DUMP_S", "0"))
    if hang_after > 0:  # where is every rank, should the run stop making progress?
        import faulthandler

        faulthandler.dump_traceback_later(hang_after, exit=True)
    torch.cuda.is_available = lambda: True
    torch.cuda.set_device = lambda *_a, **_k: None
    torch.cuda.synchronize = lambda *_a, **_k: None
    torch.cuda.empty_cache = lambda: None
    torch.cuda.Event = _Event
    torch.cuda.current_stream = lambda *_a, **_k: _Stream()
    import cpu_double
    from modin_b200 import hostpath

    hostpath.pinned_array = lambda nrows, dtype=np.float64: np.empty(int(nrows), dtype=dtype)

    def stream_map(op, code, in0, out, in1=None, in2=None, s0=None, s1=None, chunk_rows=0):
        for j, (a, o) in enumerate(zip(in0, out)):
            o[:] = {"affine": lambda: a * s0[j] + s1[j], "abs": lambda: np.abs(a), "neg": lambda: -a,
                    "add_s": lambda: a + s0[j], "mul_s": lambda: a * s0[j], "sub_s": lambda: a - s0[j],
                    "rsub_s": lambda: s0[j] - a, "div_s": lambda: a / s0[j], "rdiv_s": lambda: s0[j] / a}[op]()  # fmt: skip

    hostpath.stream_map = stream_map
    import bench

    sys.argv = [sys.argv[0]] + [a for a in sys.argv[1:]]
    args = bench.parse_args()
    args.skip_cpu = True
    with cpu_double.installed():
        from modin_b200 import config

        config.HostStreamMinBytes.put(1 << 12)  # tiny frames still take the host-streaming path
        bench.run_b200_arm(args)


if __name__ == "__main__":
    main()
