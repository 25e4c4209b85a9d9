"""CPU-only tests: the C-ABI library loads and exports every declared symbol, host-side partition
logic (chunk sizes, call-queue fusion, template wiring), the numpy generator twin, and the loud
failure when no GPU is present.  No kernel is launched here."""

import ctypes
import os
import re

import numpy as np
import pandas
import pytest

from modin_b200 import _lib, build, synth
from modin_b200.functors import DevAffine, DevBinary, DevMap
from modin_b200.partitioning import (
    B200Partition,
    Bound,
    compute_chunksize,
    fuse_call_queue,
    get_length_list,
    unwrap,
)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "modin_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mb200_[a-z0-9_]+)\s*\(", text)))


def test_library_builds_and_exports_every_declared_symbol():
    path = build.build()
    assert os.path.exists(path)
    lib = ctypes.CDLL(path)
    declared = _declared_symbols()
    assert len(declared) >= 35
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/modin_b200.h but not exported"
    # the ctypes binding covers exactly the declared surface
    assert sorted(_lib.EXPORTED_SYMBOLS) == declared


def test_binding_loads_and_reports_abi():
    lib = _lib.load()
    assert lib.mb200_abi_version() == _lib.ABI_VERSION
    assert lib.mb200_launch_count() >= 0
    assert lib.mb200_reduce_scratch_bytes(8) > 0
    assert lib.mb200_sort_scratch_bytes(1000) >= 16000


def test_no_gpu_means_loud_failure_not_fallback():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = _lib.load()
    assert lib.mb200_device_check(0) != 0
    assert b"no CPU fallback" in lib.mb200_last_error() or b"CUDA" in lib.mb200_last_error()
    import modin_b200.pandas as bpd

    with pytest.raises(_lib.B200Error):
        bpd.DataFrame(pandas.DataFrame({"a": [1.0, 2.0]}))


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "modin_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f"{f} reaches into oracle/"


def test_chunk_sizes_follow_reference_rule():
    # modin/core/storage_formats/pandas/utils.py:28-58, 156-182
    assert compute_chunksize(1_000_000, 8, 32) == 125_000
    assert compute_chunksize(10, 8, 32) == 32
    assert get_length_list(100, 4, 32) == [32, 32, 32, 4]
    assert get_length_list(64, 4, 32) == [32, 32, 0, 0]
    with pytest.raises(ValueError):
        compute_chunksize(10, 2, 0)


def test_bound_is_transparent():
    f = Bound(lambda x, y, z=0: (x, y, z), (2,), {"z": 3})
    assert f(1) == (1, 2, 3)
    fn, args, kwargs = unwrap(f)
    assert args == (2,) and kwargs == {"z": 3}
    assert unwrap(len) == (len, (), {})


def test_call_queue_fuses_mul_add_into_affine():
    q = [[DevBinary("mul"), (1.25,), {"axis": "columns", "level": None, "fill_value": None}],
         [DevBinary("add"), (0.5,), {"axis": "columns", "level": None, "fill_value": None}]]  # fmt: skip
    fused = fuse_call_queue(q)
    assert len(fused) == 1 and isinstance(fused[0][0], DevAffine)
    assert fused[0][0].mul == 1.25 and fused[0][0].add == 0.5
    # row vectors fuse too
    q2 = [[DevBinary("mul"), ([1.0, 2.0],), {}], [DevBinary("add"), ([3.0, 4.0],), {}]]
    assert isinstance(fuse_call_queue(q2)[0][0], DevAffine)
    # add then mul must NOT fuse (different arithmetic)
    q3 = [[DevBinary("add"), (1.0,), {}], [DevBinary("mul"), (2.0,), {}]]
    assert len(fuse_call_queue(q3)) == 2
    # fill_value changes semantics -> no fusion
    q4 = [[DevBinary("mul"), (1.0,), {"fill_value": 0.0}], [DevBinary("add"), (2.0,), {}]]
    assert len(fuse_call_queue(q4)) == 2
    # unrelated entries pass through
    q5 = [[DevMap("abs"), (), {}], [DevBinary("mul"), (2.0,), {}], [DevBinary("add"), (1.0,), {}]]
    out = fuse_call_queue(q5)
    assert len(out) == 2 and isinstance(out[1][0], DevAffine)


def test_call_queue_fuses_frame_mul_add_into_fma3():
    b = B200Partition(object())
    c = B200Partition(object())
    q = [[Bound(DevBinary("mul"), (), {}), (b,), {}], [Bound(DevBinary("add"), (), {}), (c,), {}]]
    fused = fuse_call_queue(q)
    assert len(fused) == 1 and fused[0][0].op == "fma3"


def test_lazy_partition_queue_is_immutable_value():
    p = B200Partition("payload")
    q = p.add_to_apply_calls(DevBinary("mul"), 2.0)
    assert p.call_queue == [] and len(q.call_queue) == 1 and q._data == "payload"


def test_synth_generators_are_deterministic_and_range_consistent():
    a = synth.gen_f64(1000, 42, 3)
    b = synth.gen_f64(400, 42, 3, row_offset=600)
    assert np.array_equal(a[600:].view(np.uint64), b.view(np.uint64))
    assert abs(a.mean()) < 0.2 and 0.8 < a.std() < 1.2
    k = synth.gen_i64(10000, 43, 0, 37)
    assert k.min() >= 0 and k.max() < 37 and len(np.unique(k)) == 37
    x = synth.gen_f64(1 << 16, 1, 0, nan_per_64k=6554)
    assert 0.05 < np.isnan(x).mean() < 0.15
    # known-answer vector (also checked against the CUDA generator in the gpu tests)
    assert synth.gen_i64(4, 43, 0, 1000).tolist() == [236, 8, 706, 2]


def test_templates_register_like_the_reference():
    from modin_b200.algebra import Map, Operator, TreeReduce

    with pytest.raises(ValueError):
        Map()
    assert Operator.validate_axis(None) == 0
    caller = TreeReduce.register(lambda x: x)
    assert callable(caller)


def test_config_parameters():
    from modin_b200 import config

    old = config.NPartitions.get()
    config.NPartitions.put(4)
    assert config.NPartitions.get() == 4
    with pytest.raises(ValueError):
        config.NPartitions.put(0)
    config.NPartitions.put(old)
    assert config.MinRowPartitionSize.get() == 32


def test_dense_table_and_skew_decisions():
    """Host-side rules that pick the table form (ops.dense_range_ok) and the hot-group cache (ops.keys_are_skewed)."""
    from modin_b200 import _lib, ops

    S = _lib.GB_SUM
    assert ops.dense_range_ok(0, 999_999, 1 << 20, 10**9, 8, S)  # the benchmark: keys in [0, 1e6)
    assert ops.dense_range_ok(-5, 5, 1024, 11, 3, S)  # tiny frames: range <= 65536 is always fine
    assert not ops.dense_range_ok(0, 10**12, 1 << 20, 10**9, 8, S)  # ids spread over a huge range -> hash table
    assert not ops.dense_range_ok(0, (1 << 29) + 1, 1 << 30, 10**10, 1, S)  # above the 2^29 group-id space
    assert ops.dense_range_ok(0, 10**8, 1 << 20, 10**9, 1, S)  # range <= rows / 2 ...
    assert not ops.dense_range_ok(0, 10**8, 1 << 20, 10**9, 32, S | _lib.GB_COUNT)  # ... unless the arrays pass 8 GiB
    # skew: share of sampled keys that met their own value among 32 keys; uniform over G keys ~ 31 / G
    assert not ops.keys_are_skewed(10**6, 31 * 10**6 // 4000)  # uniform, G = 4000 (below the shared-memory limit anyway)
    assert ops.keys_are_skewed(10**6, 276_000)  # the Zipf-like generator: 27.6 %
    assert not ops.keys_are_skewed(512, 500)  # too few samples to say anything


def test_skewed_generator_is_heavy_headed_and_reproducible():
    from modin_b200 import synth

    a = synth.gen_i64_skew(200_000, 43, 0, 1_000_000)
    assert np.array_equal(a[1000:2000], synth.gen_i64_skew(1000, 43, 0, 1_000_000, row_offset=1000))
    assert a.min() == 0 and a.max() < 1_000_000
    share0 = (a == 0).mean()
    assert 0.08 < share0 < 0.2
    top = np.sort(np.bincount(a[a < 4096], minlength=4096))[::-1]
    assert top[:256].sum() / len(a) > 0.5  # the 256 hottest keys carry more than half of the rows
    lv = synth.skew_levels(1_000_000)
    assert len(lv) == 21 and int(lv[-1]) < 2**31 and np.all(np.diff(lv.astype(np.int64)) > 0)


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs next to the GPU arm) on a tiny sample."""
    import json
    import subprocess
    import sys

    if not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "modin")):
        pytest.skip("reference Modin not installed under oracle/_ref: the reference arm has nothing to time")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-rows", "200000"], capture_output=True, text=True, timeout=300, cwd=ROOT)  # fmt: skip
    assert out.returncode == 0, out.stderr[-2000:]
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1]
    j = json.loads(line)
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "dtype", "data", "config", "cpu_baseline", "e2e"):  # fmt: skip
        assert key in j, key
    assert j["impl"] == "reference" and j["value"] > 0 and j["cpu_baseline"]["kind"] == "reference"
    assert "modin.pandas" in j["config"]["api"] and j["cpu_baseline"]["alongside"]["groupby_sum"]["checked"]
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["d2h_bytes_per_step"] == 0


def test_cum_entry_points_validate_arguments_before_touching_a_device():
    """The Fold kernels' entry points (csrc/cum.cu): scratch sizing is host arithmetic (one 8-byte aggregate per column
    and 4096-row tile), and bad arguments are refused with a message before any device is looked for -- so this runs in
    a container without a GPU."""
    import ctypes as C

    lib = _lib.load()
    assert lib.mb200_cum_scratch_bytes(8, 10**9) == 8 * ((10**9 + 4095) // 4096) * 8 + 256
    assert lib.mb200_cum_scratch_bytes(3, 0) == 3 * 8 + 256 and lib.mb200_cum_scratch_bytes(1, 4096) == 8 + 256
    none = _lib.ptr_array([None])
    for args, needle in (
        ((99, _lib.F64, 1, none, 10, None, 0, None, None), b"op must be"),
        ((_lib.CUM["ffill"], _lib.I64, 1, none, 10, None, 0, None, None), b"op must be"),
        ((_lib.CUM["sum"], _lib.U8, 1, none, 10, None, 0, None, None), b"dtype must be"),
        ((_lib.CUM["sum"], _lib.F64, -1, none, 10, None, 0, None, None), b"negative"),
        ((_lib.CUM["sum"], _lib.F64, 1, none, 10, None, 0, None, None), b"null or misaligned column"),
    ):
        assert lib.mb200_cum_partials(*args) != 0 and needle in lib.mb200_last_error(), (args[:3], lib.mb200_last_error())
    buf = (C.c_double * 4)()
    misaligned = _lib.ptr_array([C.addressof(buf) + 4])
    assert lib.mb200_cum_partials(_lib.CUM["max"], _lib.F64, 1, misaligned, 2, None, 0, None, None) != 0
    assert b"misaligned" in lib.mb200_last_error()
    assert lib.mb200_cum_carry(_lib.CUM["sum"], _lib.F64, 2, None, 1, None, None) != 0 and b"null argument" in lib.mb200_last_error()
    assert lib.mb200_cum_carry(_lib.CUM["sum"], _lib.F64, 0, None, 0, None, None) == 0  # nothing to do is not an error
