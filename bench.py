#!/usr/bin/env python
"""bench.py -- headline measurement of the B200 partition-execution path.

    python bench.py --gpus N --steps K --warmup W            # this repo's arm
    python bench.py --impl reference --gpus N --steps K --warmup W

Front door: the REAL ``modin.pandas`` with this repo's execution plugged in (``modin_b200.modin_plugin``;
Modin itself comes from ``oracle/_ref``, which ``build()`` installs from the original project) -- ``config.api`` says so.
``--api mirror`` (and the automatic fallback when Modin is not importable) uses the repo's own Modin-free mirror
of the same class protocol, ``modin_b200.pandas``.

Workload of the headline (BASELINE.json configs[1]): Map / Binary template, ``a * b + c`` over a synthetic
1e9-row x 8-column float64 frame (``a`` device resident, ``b``, ``c`` scalars -> one fused AFFINE sweep, two
IEEE roundings).  N > 1 (torchrun, one rank per GPU, NCCL): the SAME 1e9 rows are sharded row-wise over the
ranks ("strong" scaling, as the north-star's ">= 6x at 8 GPUs" is phrased).

One JSON line on rank 0:
  value            rows/s, inputs resident in HBM (CUDA events, max over ranks)
  roofline         algorithmic bytes / launch time against MEASURED_PEAKS.json (map kernel)
  roofline_groupby the same for ``groupby('key').sum()`` (BASELINE.json's other half of the metric)
  e2e              rows/s through the public API with HOST buffers: ``pd.DataFrame(host) * b + c -> _to_pandas()``
                   (pinned host in, H2D, kernel, D2H, pinned host out, all inside the timed call)
  e2e_groupby      ``pd.DataFrame(host).groupby('key').sum()._to_pandas()`` the same way (72 B/row H2D, result D2H)
  cpu_baseline     the reference's own CPU path on this box's host cores (bounded sample)
  also             the other hot-path templates measured the same way (C3 sum / mean at 16 columns, three-frame
                   a*b+c, groupby on dense / hashed / skewed keys, broadcast merge)
  every leg carries ``checked`` (its result was verified OUTSIDE the timed region); N > 1 adds ``parity_ok``
  (the hot path checked against pandas on a small job-wide frame over the NCCL group before anything is timed).

``--dump-outputs DIR`` writes what the timed steps of each leg computed in their last step as ``DIR/<name>.npy``
(float64; rows of large results at fixed seeded positions, with those positions as ``<name>_rows`` / ``<name>_index``),
so that two builds can be compared output for output on identical inputs.  Groupby sums accumulate with float
atomics and match from run to run only within the sum tolerance; every other output repeats bit for bit.

``--impl reference`` times the UNMODIFIED reference (``modin.pandas`` from ``oracle/_ref``, its own
PandasOnPython engine -- PandasOnRay when ``ray`` is importable) on a bounded sample of the same workload; rank 0
only.
"""

from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
REF = os.path.join(ROOT, "oracle", "_ref")

METRIC = "rows/sec elementwise map (a*b+c) on 1e9x8 f64"
UNIT = "rows/s"
B_SCALAR, C_SCALAR = 1.000000119, 0.5
EPS = 2.0**-53
# --dump-outputs: at most 3 MB per result (sampled values + their positions); the ten sampled results plus the two
# 16-value reductions stay far below 64 MB whatever --cols is
DUMP_BYTES_PER_OUTPUT = 3 << 20
DUMP_SEED = 20_251_017


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--api", default="auto", choices=["auto", "modin", "mirror"])
    ap.add_argument("--rows", type=float, default=1e9, help="global rows of the synthetic frame")
    ap.add_argument("--cols", type=int, default=8)
    ap.add_argument("--groups", type=int, default=1_000_000)
    ap.add_argument("--cpu-rows", type=float, default=0, help="rows of the bounded CPU sample (0 = sized to a time budget)")
    ap.add_argument("--cpu-budget", type=float, default=150.0, help="seconds the reference arm's map leg may take")
    ap.add_argument("--e2e-rows", type=float, default=1e8, help="rows of the host-buffer e2e sample (all ranks together)")
    ap.add_argument("--skip-also", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write each leg's result of its last timed step to DIR/<name>.npy (rank 0's shard when N > 1)")
    return ap.parse_args()


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_for(kernel: str, rows_local: int = 0):
    """DRAM bytes per launch of `kernel`, from the committed `ncu --set full` capture (profiles/traffic.json, taken at
    2^27 rows) scaled linearly to this run's local row count; None when no capture exists for the kernel."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        ent = t.get(kernel)
        return float(ent["dram_bytes"]) * (rows_local / float(t["rows"])) if ent else None
    except Exception:
        return None


def dump_positions(n: int, ncols: int):
    """Rows kept of an n-row, ncols-column result: all of them when they fit DUMP_BYTES_PER_OUTPUT, else the first and
    the last row and a seeded draw -- the same positions for the same shape in every run."""
    import numpy as np

    k = max(2, DUMP_BYTES_PER_OUTPUT // (8 * (ncols + 1)))
    if n <= k:
        return np.arange(n, dtype=np.int64)
    draw = np.random.default_rng(DUMP_SEED).integers(0, n, k - 2)
    return np.unique(np.concatenate([np.array([0, n - 1], dtype=np.int64), draw]))


def modin_importable() -> bool:
    return os.path.isdir(os.path.join(REF, "modin"))


# ------------------------------------------------------------------------------------ reference arm (CPU)
_MALLOC_ENV = {
    # keep big numpy buffers inside the heap and never trim it: without this every pandas temporary is a
    # fresh mmap whose first touch page-faults, which would sandbag the CPU arm by 2-10x
    "MALLOC_MMAP_THRESHOLD_": str(1 << 25),
    "MALLOC_TRIM_THRESHOLD_": str(1 << 40),
    "MALLOC_TOP_PAD_": str(1 << 28),
}


def _reference_modin():
    """``modin.pandas`` of the UNMODIFIED reference (oracle/_ref) on its own CPU engine; (module, engine name)."""
    if REF not in sys.path:
        sys.path.insert(0, REF)
    from modin_b200.modin_plugin import apply_pandas3_shims

    apply_pandas3_shims()  # the image ships pandas 3; the reference pins < 2.4 (SURVEY 8c: five removed names)
    engine = "python"
    try:
        import ray  # noqa: F401

        engine = "ray"
    except Exception:
        pass
    os.environ["MODIN_ENGINE"] = engine
    import modin.config as cfg
    import modin.pandas as mpd

    cfg.Engine.put(engine.capitalize() if engine != "python" else "Python")
    return mpd, ("PandasOnRay" if engine == "ray" else "PandasOnPython"), int(cfg.NPartitions.get())


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if os.environ.get("MB200_REF_CHILD") != "1":
        env = dict(os.environ, MB200_REF_CHILD="1", **_MALLOC_ENV)
        os.execve(sys.executable, [sys.executable] + sys.argv, env)
    import warnings

    warnings.filterwarnings("ignore")
    from modin_b200 import synth

    ncpu = os.cpu_count() or 1
    if not modin_importable():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/modin is not installed on this box"}), flush=True)
        return
    mpd, engine, nparts = _reference_modin()
    cores = 1 if engine == "PandasOnPython" else ncpu
    W = args.cols

    def modin_map_pass(mdf):
        t0 = time.perf_counter()
        out = mdf * B_SCALAR + C_SCALAR
        out._query_compiler.execute()
        dt = time.perf_counter() - t0
        assert out.shape == mdf.shape
        return dt

    # size the sample to the time budget: probe at 2e7 rows (large enough that every pandas temporary is a fresh
    # mmap, as at the real size), then scale
    total_steps = args.steps + max(args.warmup, 1)
    if args.cpu_rows:
        rows = int(args.cpu_rows)
    else:
        probe_n = 20_000_000
        probe = mpd.DataFrame(synth.host_frame(probe_n, W, seed=42))
        probe._query_compiler.execute()
        modin_map_pass(probe)
        rate = probe_n / modin_map_pass(probe)
        del probe
        rows = int(min(1e8, max(1e7, rate * args.cpu_budget / total_steps)))
    pdf = synth.host_frame(rows, W, seed=42)
    mdf = mpd.DataFrame(pdf)
    mdf._query_compiler.execute()
    for _ in range(max(args.warmup, 1)):
        modin_map_pass(mdf)
    times = [modin_map_pass(mdf) for _ in range(args.steps)]
    ms = statistics.mean(times) * 1e3
    value = rows / (ms / 1e3)
    # alongside: plain pandas on the same frame (one core), and the groupby half of the metric on a smaller sample
    t0 = time.perf_counter()
    _ = pdf * B_SCALAR + C_SCALAR
    pandas_map = rows / (time.perf_counter() - t0)
    del _, mdf, pdf
    grows = int(min(rows, 1e7))
    gpdf = synth.host_frame(grows, W, seed=42, key_modulus=args.groups)
    gm = mpd.DataFrame(gpdf)
    gm._query_compiler.execute()

    def modin_gb_pass():
        t0 = time.perf_counter()
        r = gm.groupby("key").sum()
        r._query_compiler.execute()
        return time.perf_counter() - t0, r

    modin_gb_pass()
    gdt, gres = modin_gb_pass()
    t0 = time.perf_counter()
    pres = gpdf.groupby("key").sum()
    pandas_gb = grows / (time.perf_counter() - t0)
    gb_checked = bool(len(gres) == len(pres))
    line = {
        "impl": "reference",
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"map_partitions elementwise a*b+c (b,c scalars) on {int(args.rows)}x{W} f64 -- reference "
                               f"arm: a {rows}x{W} sample of it per step",
                   "rows": int(args.rows), "cols": W, "sample_rows": rows,
                   "api": f"modin.pandas ({engine}, unmodified reference from oracle/_ref, pandas-3 import shims)",
                   "npartitions": nparts},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference", "engine": engine,
                         "host_cores": ncpu,
                         "sample": f"{rows} rows x {W} cols per step, {args.steps} steps",
                         "alongside": {"plain_pandas_1core_rows_s": pandas_map,
                                       "groupby_sum": {"rows": grows, "groups": args.groups,
                                                       "modin_rows_s": grows / gdt, "plain_pandas_rows_s": pandas_gb,
                                                       "checked": gb_checked}}},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }  # fmt: skip
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------ GPU arm
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")  # fmt: skip

    def __init__(self, device_index: int):
        self.idx = device_index
        self.file = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.idx)], stdout=self.file, stderr=subprocess.DEVNULL)  # fmt: skip
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        self.file.flush()
        rows = []
        try:
            with open(self.file.name) as fh:
                for ln in fh:
                    parts = [p.strip() for p in ln.split(",")]
                    if len(parts) >= 9:
                        rows.append(parts)
        finally:
            try:
                os.unlink(self.file.name)
            except OSError:
                pass
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = [float(r[1]) for r in rows if r[1].replace(".", "", 1).isdigit()]
        mx = [float(r[2]) for r in rows if r[2].replace(".", "", 1).isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            for name, val in zip(names, r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        # the median over samples taken while the GPU was actually clocked up (idle samples sit at the floor)
        busy = [v for v in sm if mx and v >= 0.5 * max(mx)] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(rows)}  # fmt: skip


class Api:
    """The front door the legs are driven through: real ``modin.pandas`` with the B200 execution plugged in, or the
    repo's Modin-free mirror.  Both hand out pandas-style frames with ``_query_compiler`` / ``_to_pandas()``."""

    def __init__(self, which: str):
        from modin_b200 import synth

        self.synth = synth
        if which == "auto":
            which = "modin" if modin_importable() else "mirror"
        self.which = which
        if which == "modin":
            if REF not in sys.path:
                sys.path.insert(0, REF)
            import warnings

            warnings.filterwarnings("ignore")
            from modin_b200 import modin_plugin

            self.plugin = modin_plugin
            modin_plugin.activate()
            import modin.config as cfg
            import modin.pandas as mpd

            cfg.NPartitions.put(1)
            self.pd = mpd
            self.name = "modin.pandas (ArrowOnB200: real Modin from oracle/_ref + modin_b200.modin_plugin)"
        else:
            import modin_b200.pandas as bpd

            self.pd = bpd
            self.name = "modin_b200.pandas (Modin-free mirror of the class protocol)"

    def device_frame(self, rows, W, **kw):
        """This rank's shard of the synthetic frame, generated in HBM (from_map-style ingest: no host frame)."""
        if self.which == "modin":
            return self.plugin.from_device_blocks(self.synth.device_blocks(rows, W, npartitions=1, **kw))
        return self.synth.device_frame(rows, W, npartitions=1, **kw)

    @staticmethod
    def execute(obj):
        qc = getattr(obj, "_query_compiler", None)
        if qc is not None:
            qc.execute()
        return obj

    @staticmethod
    def launch(obj):
        """Run the frame's pending work WITHOUT waiting for the device: ``qc.finalize()`` drains the call queues
        (= launches the kernels on the rank's stream); ``qc.execute()`` would add ``wait_computations``.  The timed
        region is bracketed by device synchronisations, the steps inside it are not -- the host prepares step i + 1
        while the GPU runs step i, as any asynchronous engine is used."""
        qc = getattr(obj, "_query_compiler", None)
        if qc is not None:
            qc.finalize()
        return obj

    def cumsum(self, obj):
        """``df.cumsum()``; the mirror's API layer has no Fold methods, so there the query compiler's is called."""
        if self.which == "modin":
            return obj.cumsum()
        return self.pd.DataFrame(query_compiler=obj._query_compiler.cumsum(0))

    @staticmethod
    def to_pandas(obj):
        return obj._to_pandas() if hasattr(obj, "_to_pandas") else obj

    @staticmethod
    def blocks(obj):
        """This rank's device blocks of a frame, one per row partition (first column partition)."""
        return [row[0].get() for row in obj._query_compiler._modin_frame._partitions]


def _bits_equal(a, b):
    import numpy as np

    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and bool(((a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))).all())


def _sum_close(got, want, abs_sum, n):
    import numpy as np

    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    tol = 4.0 * max(1.0, math.log2(max(n, 2))) * EPS * np.asarray(abs_sum, dtype=np.float64) + 1e-300
    return got.shape == want.shape and bool((np.abs(got - want) <= tol).all())


def parity_over_ranks(api: Api):
    """The hot path on a small JOB-WIDE frame (every rank ingests its shard of the same seeded host frame), gathered
    and compared with pandas on the whole frame: bit-exact for elementwise / count / min / max / keys / merge, the
    stated sum tolerance for sums and means.  Returns (ok, failed check names).  Runs before anything is timed."""
    import numpy as np
    import pandas

    from modin_b200 import config as _cfg
    from modin_b200 import synth

    fails = []

    def check(name, ok):
        if not ok:
            fails.append(name)

    n, W, G = 100_003, 4, 2_003
    pdf = synth.host_frame(n, W, seed=42, nan_per_64k=700, key_modulus=G)
    vals = pdf.drop(columns="key")
    P = api.to_pandas
    df, dv = api.pd.DataFrame(pdf), api.pd.DataFrame(vals)
    check("map abs", _bits_equal(P(dv.abs()).to_numpy(), vals.abs().to_numpy()))
    check("fused a*b+c", _bits_equal(P(dv * 1.25 + 0.5).to_numpy(), (vals * 1.25 + 0.5).to_numpy()))
    abs_sum = np.nansum(np.abs(vals.to_numpy()), axis=0)
    check("tree_reduce sum", _sum_close(np.asarray(P(dv.sum())), vals.sum().to_numpy(), abs_sum, n))
    check("tree_reduce count", np.array_equal(np.asarray(P(dv.count())), vals.count().to_numpy()))
    check("tree_reduce min", _bits_equal(np.asarray(P(dv.min())), vals.min().to_numpy()))
    check("tree_reduce mean", _sum_close(np.asarray(P(dv.mean())), vals.mean().to_numpy(),
                                         abs_sum / np.maximum(vals.count().to_numpy(), 1), n))  # fmt: skip
    gabs = vals.abs().groupby(pdf["key"]).sum().to_numpy()
    want = pdf.groupby("key").sum()
    for dense in (True, False):
        _cfg.GroupbyDenseKeys.put(dense)
        tag = "dense" if dense else "hash"
        got = P(df.groupby("key").sum())
        check(f"groupby[{tag}] keys", np.array_equal(got.index.to_numpy(), want.index.to_numpy()))
        check(f"groupby[{tag}] sum", got.shape == want.shape and _sum_close(got.to_numpy(), want.to_numpy(), gabs, n))
        check(f"groupby[{tag}] count", np.array_equal(P(df.groupby("key").count()).to_numpy(), pdf.groupby("key").count().to_numpy()))
    _cfg.GroupbyDenseKeys.put(True)
    rng = np.random.RandomState(5)
    dim = pandas.DataFrame({"key": rng.permutation(G).astype(np.int64)[: int(G * 0.9)]})
    dim["d0"] = synth.gen_f64(len(dim), 11, 0)
    left = P(df.merge(api.pd.DataFrame(dim), on="key", how="left"))
    wl = pdf.merge(dim, on="key", how="left")
    check("merge left", list(left.columns) == list(wl.columns) and _bits_equal(left.to_numpy(dtype=np.float64), wl.to_numpy(dtype=np.float64)))
    return (not fails), fails


def run_b200_arm(args):
    import numpy as np
    import pandas
    import torch

    from modin_b200 import _lib, dist, synth
    from modin_b200 import config as _cfg
    from modin_b200.config import NPartitions

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 arm has no CPU fallback")
    # DEV / backend are "cuda" / "nccl" in every real run; tests/bench_dryrun.py swaps the device for the numpy double
    # (and torch.cuda.* for stand-ins) to run this function's control flow under gloo at world sizes no CPU box has GPUs for
    DEV = os.environ.get("MB200_BENCH_DEVICE", "cuda")
    distributed = dist.init_from_env("nccl" if DEV == "cuda" else "gloo")
    ws, rank = dist.world_size(), dist.rank()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    lib = _lib.load()
    if DEV == "cuda":
        _lib.check(lib.mb200_device_check(local))
    NPartitions.put(1)
    hbm_peak, peak_src = measured_peaks()
    api = Api(args.api)

    def progress(msg):
        """One line per leg on stderr (rank 0): where a run is, should it ever stop making progress."""
        if rank == 0:
            print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


    def release():
        """Between legs: collect cyclic garbage first (Modin's API objects reference themselves; a dead 32 GB result
        held by such a cycle would survive ``empty_cache``), then hand the cached blocks back to the driver."""
        import gc

        gc.collect()
        torch.cuda.empty_cache()

    rows, W, G = int(args.rows), args.cols, args.groups
    lo, hi = dist.shard_bounds(rows)
    rows_local = hi - lo

    def sync_all():
        torch.cuda.synchronize()
        if distributed:
            torch.distributed.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if not distributed:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=DEV)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    def all_ranks_ok(ok: bool) -> bool:
        if not distributed:
            return bool(ok)
        t = torch.tensor([0 if ok else 1], dtype=torch.int64, device=DEV)
        torch.distributed.all_reduce(t)
        return int(t.item()) == 0

    def timed(step_fn, steps, warmup):
        """W untimed steps, then exactly K steps between barrier+sync, CUDA events on the launching
        stream; returns (total ms max over ranks, per-step ms list on this rank)."""
        import gc

        for _ in range(warmup):
            step_fn()
        gc.collect()  # like timeit: a generation-2 collection (tens of ms with Modin's object graphs alive) must not
        gc.disable()  # land inside a 3 ms step; the collector runs again as soon as the timed steps are launched
        sync_all()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        evs[0].record()
        try:
            for i in range(steps):
                step_fn()
                evs[i + 1].record()
        finally:
            gc.enable()
        torch.cuda.synchronize()
        per = [evs[i].elapsed_time(evs[i + 1]) for i in range(steps)]
        total = evs[0].elapsed_time(evs[steps])
        sync_all()
        return max_over_ranks(total), per

    from modin_b200 import ops as _ops

    def kernel_ms(step_fn, tag, reps=3):
        """Average duration of ONE launch of the dominant kernel (CUDA events around the C call on the launching
        stream, ops.KernelTimer), over `reps` extra steps run after the timed region; max over ranks."""
        with _ops.KernelTimer() as kt:
            for _ in range(reps):
                step_fn()
            ms = kt.total_ms(tag)
        sync_all()
        # per step: a template may launch the kernel more than once (map phase + the tiny reduce phase over the
        # partials); the step's launches are added up, so the figure is the time the step spends in this kernel
        return max_over_ranks(ms / reps) if ms is not None else None

    def roof(kernel, bytes_per_launch_local, per_ms, traffic=None, launch_ms=None, **extra):
        """`achieved` = algorithmic bytes of one launch / that kernel's own duration (`launch_ms`, CUDA events around
        the launch); `step_frac` is the same bytes over the WHOLE step (API layer, small kernels, collectives)."""
        step = statistics.mean(per_ms)
        lm = launch_ms if launch_ms else step
        ach = bytes_per_launch_local / (lm / 1e3) / 1e9
        return {"bound": "hbm", "kernel": kernel, "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                "frac": ach / hbm_peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": bytes_per_launch_local, "launch_ms": lm, "step_ms": step,
                "per_step_ms": [round(x, 3) for x in per_ms],
                "step_frac": bytes_per_launch_local / (step / 1e3) / 1e9 / hbm_peak, **extra}  # fmt: skip

    def sample_rows(n):
        return sorted({0, 1, min(4095, n - 1), min(4096, n - 1), n // 2, n - 1}) if n > 0 else []

    def device_values(col, idx):
        return col.data[torch.tensor(idx, dtype=torch.int64, device=col.data.device)].cpu().numpy()

    dumped = {}  # --dump-outputs: name -> float64 array, kept on rank 0 and written after the last leg

    def dump(name, arr):
        if args.dump_outputs is not None and rank == 0:
            dumped[name] = np.asarray(arr, dtype=np.float64)

    def dump_block(name, frame, row0):
        """Sampled rows of this rank's device result block of ``frame``, and their positions in the whole frame."""
        if args.dump_outputs is not None and rank == 0:
            blk = api.blocks(frame)[0]
            idx = dump_positions(blk.nrows, len(blk.cols))
            dump(name, np.stack([device_values(c, idx) for c in blk.cols], axis=1))
            dump(name + "_rows", idx + row0)

    def dump_frame(name, frame):
        """Sampled rows of a host result frame, and its index at those rows."""
        if args.dump_outputs is not None and rank == 0:
            idx = dump_positions(len(frame), frame.shape[1])
            dump(name, frame.iloc[idx].to_numpy(dtype=np.float64))
            dump(name + "_index", frame.index.to_numpy()[idx])

    # ---- multi-GPU parity before anything is timed ------------------------------------------------
    parity_ok, parity_fails = None, []
    progress(f"start: {ws} rank(s), {rows} rows, front door {api.which}")
    if distributed:
        try:
            ok, parity_fails = parity_over_ranks(api)
        except Exception as exc:  # a crash is a failed check, on every rank
            ok, parity_fails = False, [f"{type(exc).__name__}: {exc}"[:300]]
        parity_ok = all_ranks_ok(ok)

    # ---- headline: fused a*b+c through the public API ---------------------------------------
    progress(f"parity_ok={parity_ok}; headline map")
    a = api.device_frame(rows, W, seed=42)
    api.execute(a)
    last = [None]

    def step_map():
        last[0] = None  # the previous result (64 GB at 1e9 rows) goes back to the allocator first
        out = a * B_SCALAR + C_SCALAR  # Binary template x2 -> call queue -> one AFFINE sweep
        api.launch(out)
        last[0] = out

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    step_map()
    launches0 = lib.mb200_launch_count()
    total_ms, per = timed(step_map, args.steps, args.warmup)
    dump_block("map_abc", last[0], lo)
    launches = lib.mb200_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    launches_timed = round(launches * args.steps / max(args.steps + args.warmup, 1))
    if distributed:
        t = torch.tensor([launches_timed], dtype=torch.int64, device=DEV)
        torch.distributed.all_reduce(t)
        launches_timed = int(t.item())
    ms_per_step = total_ms / args.steps
    value = rows / (ms_per_step / 1e3)
    roofline = roof("map_kernel<AFFINE,f64> (256-bit column sweep)", rows_local * W * 16, per,
                    traffic_for("map_affine", rows_local), launch_ms=kernel_ms(step_map, "map_affine"))  # fmt: skip
    # check (outside the timed region): sampled rows against the numpy twin of the generator, bit for bit
    blk = api.blocks(last[0])[0]
    idx = sample_rows(blk.nrows)
    ok = blk.nrows == rows_local
    for j in (0, W - 1):
        ref = np.array([synth.gen_f64(1, 42, j, lo + r)[0] for r in idx]) * B_SCALAR + C_SCALAR
        ok = ok and _bits_equal(device_values(blk.cols[j], idx), ref)
    map_checked = all_ranks_ok(ok)
    last[0] = None
    del blk  # the block is the 64 GB result: drop the last reference before the next leg allocates

    also = []
    roofline_groupby = None

    def _secondary_legs():
        nonlocal a, roofline_groupby
        ksteps = args.steps
        cols8 = [f"c{j}" for j in range(W)]
        # sums of the headline frame with the direct-load reduce kernel: the cross-check value for the TMA kernel below
        _cfg.ReduceVariant.put(1)
        sum8_ldg = np.asarray(api.to_pandas(a.sum()), dtype=np.float64)
        _cfg.ReduceVariant.put(0)
        abs8 = np.asarray(api.to_pandas(a.abs().sum()), dtype=np.float64)
        a = None
        release()

        progress("leg: TreeReduce sum / mean, 16 columns")
        # ---- TreeReduce (C3): df.sum() / df.mean() over 16 float64 columns.  1e9 x 16 f64 = 128 GB: the whole frame
        # on one 180 GB B200, 16 GB per GPU at 8
        W3 = 16
        c3 = api.device_frame(rows, W3, seed=42)
        api.execute(c3)
        res = {}

        def step_sum():
            res["sum"] = api.launch(c3.sum())

        def step_mean():
            res["mean"] = api.launch(c3.mean())

        for name, fn in (("sum", step_sum), ("mean", step_mean)):
            total_s, per_s = timed(fn, ksteps, 2)
            got = np.asarray(api.to_pandas(res[name]), dtype=np.float64)
            dump(f"reduce_{name}", got)
            if name == "sum":
                sum16 = got
                ok = _sum_close(got[:W], sum8_ldg, abs8, rows)  # same first 8 columns, other reduce kernel
            else:
                ok = _sum_close(got, sum16 / rows, np.concatenate([abs8, abs8])[:W3] / rows + np.abs(sum16) / rows, rows)
            also.append({"metric": f"rows/sec TreeReduce df.{name}() on 1e9x16 f64 (C3; result stays on the device)",
                         "value": rows / (total_s / ksteps / 1e3), "unit": UNIT, "ms_per_step": total_s / ksteps,
                         "checked": bool(ok),
                         "roofline": roof("reduce_tma_kernel<SUM,f64> + reduce_finalize" + (" (+ count, divide)" if name == "mean" else ""),
                                          rows_local * W3 * 8, per_s, traffic_for("reduce_sum", rows_local * 2),
                                          launch_ms=kernel_ms(fn, "reduce_sum"))})  # fmt: skip
        del c3, res
        release()

        # ---- Binary template on three frames: a*b+c with b, c frames (C2 secondary form; 256 B/row fused).
        # Four n x 8 frames are resident, so n = rows/4 (2.5e8 per 1e9: 64 GB on one GPU)
        progress("leg: three-frame a*b+c")
        rows3 = max(rows // 4, 1024)
        lo3, _hi3 = dist.shard_bounds(rows3)
        fa, fb, fc = (api.device_frame(rows3, W, seed=s) for s in (42, 44, 45))
        for f in (fa, fb, fc):
            api.execute(f)

        def step_fma3():
            last[0] = None
            out = fa * fb + fc  # two n_ary_op calls -> call queue -> one FMA3 sweep (two roundings)
            api.launch(out)
            last[0] = out

        total_f, per_f = timed(step_fma3, ksteps, 2)
        blk = api.blocks(last[0])[0]
        dump_block("map_fma3", last[0], lo3)
        idx = sample_rows(blk.nrows)
        j = W - 1
        ref = (np.array([synth.gen_f64(1, 42, j, lo3 + r)[0] for r in idx]) * np.array([synth.gen_f64(1, 44, j, lo3 + r)[0] for r in idx])
               + np.array([synth.gen_f64(1, 45, j, lo3 + r)[0] for r in idx]))  # fmt: skip
        ok = all_ranks_ok(_bits_equal(device_values(blk.cols[j], idx), ref))
        last[0] = None
        also.append({"metric": f"rows/sec a*b+c on three frames ({rows3}x8 f64 each), Binary template x2 fused",
                     "value": rows3 / (total_f / ksteps / 1e3), "unit": UNIT, "ms_per_step": total_f / ksteps, "checked": ok,
                     "roofline": roof("map_kernel<FMA3,f64>", blk.nrows * W * 32, per_f, launch_ms=kernel_ms(step_fma3, "map_fma3"))})  # fmt: skip
        del fa, fb, fc, blk
        release()

        # ---- Fold template: df.cumsum() down the rows (qc.py:2431; csrc/cum.cu).  Input + output resident, so
        # n = rows/2 (32 + 32 GB per 1e9 on one GPU); rows sharded over ranks scan locally, carries cross the ranks
        progress("leg: Fold cumsum")
        try:
            rowsf = max(rows // 2, 8192)
            lof, hif = dist.shard_bounds(rowsf)
            ff = api.device_frame(rowsf, W, seed=42)
            api.execute(ff)

            def step_cumsum():
                last[0] = None
                last[0] = api.launch(api.cumsum(ff))  # qc.cumsum -> Fold template -> frame.fold -> DevCumulative

            total_c, per_c = timed(step_cumsum, ksteps, 2)
            blk = api.blocks(last[0])[0]
            dump_block("fold_cumsum", last[0], lof)
            j = W - 1
            ok = True
            fsum = np.asarray(api.to_pandas(ff.sum()), dtype=np.float64)
            fabs = np.asarray(api.to_pandas(ff.abs().sum()), dtype=np.float64)
            try:  # rank-specific checks: whatever goes wrong here must not keep this rank from the collective below
                if rank == 0:  # the top of the frame against numpy's sequential cumsum of the same generated rows
                    m = min(blk.nrows, 10000)
                    x = synth.gen_f64(m, 42, j, 0)
                    got = blk.cols[j].data[:m].cpu().numpy()
                    ok = _sum_close(got, np.cumsum(x), np.cumsum(np.abs(x)), max(m, 2))
                if rank == ws - 1 and blk.nrows:  # the last row of the job holds the column sums (TreeReduce kernel)
                    ok = ok and _sum_close(device_values(blk.cols[j], [blk.nrows - 1]), fsum[j : j + 1], fabs[j : j + 1], rowsf)
            except Exception:
                ok = False
            ok = all_ranks_ok(ok)
            last[0] = None
            also.append({"metric": f"rows/sec df.cumsum() on {rowsf}x{W} f64, Fold template",
                         "value": rowsf / (total_c / ksteps / 1e3), "unit": UNIT, "ms_per_step": total_c / ksteps, "checked": ok,
                         "roofline": roof("cum_tile_scan_kernel<f64,SUM> (after cum_tile_reduce + cum_scan_tiles: the input is read twice, 24 B moved per 16 B algorithmic)",
                                          (hif - lof) * W * 16, per_c, launch_ms=kernel_ms(step_cumsum, "cum_apply"),
                                          partials_ms=kernel_ms(step_cumsum, "cum_partials"))})  # fmt: skip
            del ff, blk
        except Exception as exc:  # a leg added late in round 2: a failure here must not take the other legs with it
            also.append({"metric": "rows/sec df.cumsum(), Fold template", "error": f"{type(exc).__name__}: {exc}"[:300]})
        last[0] = None
        release()

        # ---- GroupByReduce: groupby('key').sum(), G int64 keys, 8 float64 values (C4)
        def groupby_leg(skew, dense_on, label, kern, traffic_key, name):
            nonlocal roofline_groupby
            progress(f"leg: groupby{label or ' dense'}")
            g = api.device_frame(rows, W, seed=42, key_modulus=G, key_skew=skew)
            api.execute(g)
            _cfg.GroupbyDenseKeys.put(dense_on)

            gb = g.groupby("key")  # the GroupBy object is built once (as pandas' own asv GroupByMethods does in setup)

            def step_gb():
                last[0] = None
                last[0] = api.launch(gb.sum())  # qc.groupby_sum -> GroupByReduce template -> frame.groupby_reduce

            def step_gb_full():  # including the API-layer construction of the GroupBy object (df[by] etc.)
                last[0] = None
                last[0] = api.launch(g.groupby("key").sum())

            try:
                total_g, per_g = timed(step_gb, ksteps, 2)
                if args.dump_outputs is not None:  # on every rank: gathering the key ranges is collective
                    dump_frame(name, api.to_pandas(last[0]))
                total_full, _ = timed(step_gb_full, ksteps, 1)
                k_ms = kernel_ms(step_gb, "gb_accumulate")
                # ---- checks, outside the timed region
                res = api.to_pandas(last[0])  # gathers every rank's key range: G x 8 (72 MB at G = 1e6)
                last[0] = None
                vals = g[cols8]
                col_sum = np.asarray(api.to_pandas(vals.sum()), dtype=np.float64)
                col_abs = np.asarray(api.to_pandas(vals.abs().sum()), dtype=np.float64)
                keys = res.index.to_numpy()
                ok = bool(len(keys) > 0 and (np.diff(keys) > 0).all() and keys[0] >= 0 and keys[-1] < G)
                if not skew:
                    ok = ok and len(keys) == min(G, rows)  # 1e9 uniform rows over 1e6 keys: every key occurs
                ok = ok and _sum_close(res.to_numpy().sum(axis=0), col_sum, col_abs, rows)
                # sampled groups against an independent device path: boolean row selection + TreeReduce
                for k in ([0, int(keys[len(keys) // 2]), int(keys[-1])] if len(keys) else []):
                    sel = g[g["key"] == k][cols8]
                    want = np.asarray(api.to_pandas(sel.sum()), dtype=np.float64)
                    wabs = np.asarray(api.to_pandas(sel.abs().sum()), dtype=np.float64)
                    pos = int(np.searchsorted(keys, k))
                    ok = ok and pos < len(keys) and keys[pos] == k and _sum_close(res.to_numpy()[pos], want, wabs, rows)
                ok = all_ranks_ok(ok)
            finally:
                _cfg.GroupbyDenseKeys.put(True)
            rf = roof(kern, rows_local * (8 + 8 * W), per_g, traffic_for(traffic_key, rows_local) if traffic_key else None,
                      launch_ms=k_ms)
            entry = {"metric": f"rows/sec groupby('key').sum() {rows} rows, {G} int64 keys{label}, 8 f64 vals",
                     "value": rows / (total_g / ksteps / 1e3), "unit": UNIT, "ms_per_step": total_g / ksteps,
                     "groups": int(len(keys)), "checked": ok, "roofline": rf,
                     "step": "gb = df.groupby('key') once; timed: gb.sum()",
                     "ms_per_step_full_expression": total_full / ksteps}  # fmt: skip
            also.append(entry)
            if not skew and dense_on:
                roofline_groupby = dict(rf, value=entry["value"], ms_per_step=entry["ms_per_step"], checked=ok,
                                        note="key range and skew flag come from statistics the generator kernel left "
                                             "on the key column (column metadata): no pre-pass over the keys")  # fmt: skip
            del g
            release()

        groupby_leg(False, True, "", "gb_accumulate_tma_kernel on a dense (direct-addressed) table pinned in L2", "groupby_sum_dense",
                    "groupby_sum_dense")
        groupby_leg(False, False, " [hash table forced]", "gb_accumulate_tma_kernel (open-addressed hash aggregate)", "groupby_sum",
                    "groupby_sum_hash")
        groupby_leg(True, True, " SKEWED (Zipf-like)", "gb_accumulate_tma_kernel<HOT> (dense table, per-CTA hot-group cache)", None,
                    "groupby_sum_skewed")
        # what a key column of UNKNOWN origin pays once: the 8 B/row statistics pass (mb200_key_range)
        from modin_b200 import ops as _ops

        kc = _ops.gen_i64(min(rows_local, 1 << 28), 43, 0, G, lo)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        _ops.key_range_device([kc])
        e0.record()
        _ops.key_range_device([kc])
        e1.record()
        torch.cuda.synchronize()
        if roofline_groupby is not None:
            roofline_groupby["key_stats_pass_ms_per_1e9_rows_unknown_column"] = e0.elapsed_time(e1) * (1e9 / len(kc))
        del kc

        # ---- broadcast merge: fact (rows x (key + 8 f64)) LEFT JOIN dim (1e7 x (key + 1 f64)) on int64 key (C5)
        progress("leg: broadcast merge")
        ndim = int(min(10_000_000, max(1000, rows // 100)))
        fact = api.device_frame(rows, W, seed=42, key_modulus=ndim)
        api.execute(fact)
        rng = np.random.RandomState(5)
        dim_keys = rng.permutation(ndim).astype(np.int64)
        d0 = synth.gen_f64(ndim, 11, 0)
        dim = api.pd.DataFrame(pandas.DataFrame({"key": dim_keys, "d0": d0}))  # sharded by rank; merge() all-gathers it
        row_of = np.empty(ndim, dtype=np.int64)
        row_of[dim_keys] = np.arange(ndim)

        def step_merge():
            last[0] = None
            last[0] = api.launch(fact.merge(dim, on="key", how="left"))

        for dense_on, label, kern in (
            (True, "", "join_dense_build + join_dense_probe (direct-addressed dim table, fused payload gather)"),
            (False, " [hash table forced]", "join_build + join_probe_gather (open-addressed hash table)"),
        ):
            if dense_on:
                os.environ.pop("MB200_JOIN_DENSE", None)
            else:
                os.environ["MB200_JOIN_DENSE"] = "0"
            try:
                total_m, per_m = timed(step_merge, ksteps, 2)
                dump_block("merge_left_" + ("dense" if dense_on else "hash"), last[0], lo)
                km_ms = kernel_ms(step_merge, "join_probe_gather")
            finally:
                os.environ.pop("MB200_JOIN_DENSE", None)
            blk = api.blocks(last[0])[0]
            idx = sample_rows(blk.nrows)
            fk = np.array([synth.gen_i64(1, 43, 0, ndim, lo + r)[0] for r in idx])
            ok = blk.nrows == rows_local and list(blk.columns) == ["key"] + cols8 + ["d0"]
            ok = ok and np.array_equal(device_values(blk.cols[0], idx), fk)
            ok = ok and _bits_equal(device_values(blk.cols[-1], idx), d0[row_of[fk]])
            ok = all_ranks_ok(ok)
            last[0] = None
            ms_m = total_m / ksteps
            moved16, moved152 = rows_local * 16, rows_local * 152
            rf = roof(kern, moved16, per_m, launch_ms=km_ms)
            rf["traffic_note"] = ("no ncu capture of the key-ordered payload probe this leg runs; the rows[] + gather "
                                  "variant moves 6.2x its algorithmic bytes (profiles/traffic.json: join_dense_gather)")
            rf["note"] = ("algorithmic bytes = 16 B/row: key read + payload written -- the fact columns of the result are "
                          "shared by reference, never copied; SURVEY 8(d) counts the reference's materialised output, "
                          "152 B/row: see frac_vs_152B_row")
            rf["frac_vs_152B_row"] = moved152 / (rf["launch_ms"] / 1e3) / 1e9 / hbm_peak
            also.append({"metric": f"rows/sec fact.merge(dim, on='key', how='left'), {rows} fact rows x {ndim} dim rows{label}",
                         "value": rows / (ms_m / 1e3), "unit": UNIT, "ms_per_step": ms_m, "checked": ok, "roofline": rf})  # fmt: skip
            del blk
        del fact, dim
        release()

    if not args.skip_also:
        try:
            _secondary_legs()
        except Exception as exc:  # a secondary leg must never cost the headline line
            import traceback

            also.append({"metric": "secondary legs aborted", "error": f"{type(exc).__name__}: {exc}"[:400],
                         "where": traceback.format_exc().strip().splitlines()[-3:]})
            os.environ.pop("MB200_JOIN_DENSE", None)
            _cfg.GroupbyDenseKeys.put(True)
            _cfg.ReduceVariant.put(0)
    a = None
    last[0] = None
    release()

    # ---- e2e: host frames in, host frames out, through the public API (rank-local sample) ----------------
    e2e = e2e_groupby = None
    progress("legs done; e2e")
    if not args.skip_e2e:
        from modin_b200 import hostpath

        er = int(args.e2e_rows) // ws

        def fill(arr, seed, col):
            m = min(len(arr), 1 << 20)
            arr[:] = np.resize(synth.gen_f64(m, seed, col), len(arr))

        def host_timed(step_fn):
            step_fn()
            sync_all()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                step_fn()
            torch.cuda.synchronize()
            return max_over_ranks((time.perf_counter() - t0) / args.steps * 1e3)

        with dist.local_frames():  # every rank runs the same host-to-host pipeline on ITS OWN host frame
            try:
                arrs = {f"c{j}": hostpath.pinned_array(er, np.float64) for j in range(W)}
                for j in range(W):
                    fill(arrs[f"c{j}"], 42, j)
                host = pandas.DataFrame(arrs, copy=False)  # columns stay the pinned buffers (no consolidation)
                out = [None]

                def step_e2e():
                    out[0] = None  # the previous result's pinned buffers go back to the pool (and are taken again below)
                    df = api.pd.DataFrame(host)  # ingest: the block stays on the host (HostBlock)
                    out[0] = api.to_pandas(df * B_SCALAR + C_SCALAR)  # streamed: H2D / AFFINE sweep / D2H per chunk

                dt = host_timed(step_e2e)
                got = out[0]
                dump_frame("e2e_map_abc", got)
                ref = host["c0"].to_numpy()[:1000] * B_SCALAR + C_SCALAR
                ok = got.shape == (er, W) and bool((got["c0"].to_numpy()[:1000] == ref).all()) and \
                    bool((got[f"c{W - 1}"].to_numpy()[-1000:] == host[f"c{W - 1}"].to_numpy()[-1000:] * B_SCALAR + C_SCALAR).all())
                e2e = {"value": er * ws / (dt / 1e3), "unit": UNIT, "h2d_bytes_per_step": er * W * 8,
                       "d2h_bytes_per_step": er * W * 8, "rows_per_step": er * ws, "ms_per_step": dt, "checked": bool(ok),
                       "path": f"{api.name}: pd.DataFrame(host) * b + c -> _to_pandas(); pinned host frame in, pooled "
                               "pinned columns out; HostBlock -> mb200_map_host (H2D / AFFINE / D2H on three streams)"}  # fmt: skip
                del got, out, host, arrs
            except Exception as exc:
                e2e = {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                       "error": f"{type(exc).__name__}: {exc}"[:300]}
            try:
                arrs = {"key": hostpath.pinned_array(er, np.int64), **{f"c{j}": hostpath.pinned_array(er, np.float64) for j in range(W)}}
                arrs["key"][:] = np.resize(synth.gen_i64(min(er, 1 << 22), 43, 0, G), er)
                for j in range(W):
                    fill(arrs[f"c{j}"], 42, j)
                host = pandas.DataFrame(arrs, copy=False)
                out = [None]

                def step_e2e_gb():
                    out[0] = None
                    df = api.pd.DataFrame(host)
                    out[0] = api.to_pandas(df.groupby("key").sum())  # H2D 72 B/row, device groupby, result D2H

                dt = host_timed(step_e2e_gb)
                got = out[0]
                dump_frame("e2e_groupby_sum", got)
                keys = host["key"].to_numpy()
                ok = len(got) == len(np.unique(keys[: 1 << 22])) if er >= (1 << 22) else True
                want0 = np.bincount(keys, weights=host["c0"].to_numpy(), minlength=G)[got.index.to_numpy()]
                wabs0 = np.bincount(keys, weights=np.abs(host["c0"].to_numpy()), minlength=G)[got.index.to_numpy()]
                ok = bool(ok) and _sum_close(got["c0"].to_numpy(), want0, wabs0, er)
                e2e_groupby = {"value": er * ws / (dt / 1e3), "unit": UNIT, "h2d_bytes_per_step": er * (8 + 8 * W),
                               "d2h_bytes_per_step": int(len(got)) * (8 + 8 * W), "rows_per_step": er * ws,
                               "ms_per_step": dt, "checked": bool(ok),
                               "path": f"{api.name}: pd.DataFrame(host).groupby('key').sum()._to_pandas()"}  # fmt: skip
                del got, out, host, arrs
            except Exception as exc:
                e2e_groupby = {"value": None, "unit": UNIT, "error": f"{type(exc).__name__}: {exc}"[:300]}
        if distributed:
            torch.distributed.barrier()

    # ---- CPU baseline (rank 0, bounded sample): the reference arm itself, in its own process ---------------
    cpu = None
    if rank == 0 and not args.skip_cpu and ws == 1:
        env = dict(os.environ, RANK="0", WORLD_SIZE="1")
        for k in ("LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT", "MB200_REF_CHILD"):
            env.pop(k, None)
        try:
            res = subprocess.run(
                [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2", "--warmup", "1",
                 "--cpu-budget", "20", "--cols", str(W), "--groups", str(G), "--rows", str(rows)]
                + (["--cpu-rows", str(int(args.cpu_rows))] if args.cpu_rows else []),
                capture_output=True, text=True, timeout=900, env=env)  # fmt: skip
            ref = json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])
            cpu = ref["cpu_baseline"]
        except Exception as e:  # the GPU numbers stand on their own; say why the CPU leg is missing
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": f"failed: {e!r}"[:300]}

    progress("done")
    if args.dump_outputs is not None and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ws, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"map_partitions elementwise a*b+c (b,c scalars, fused AFFINE, 2 roundings) on "
                                   f"{rows}x{W} f64, row-sharded over {ws} GPU(s)", "rows": rows, "cols": W,
                       "l2_policy": "inputs_larger_than_l2 (64 GB streamed per step)", "npartitions_per_gpu": 1,
                       "timing": "CUDA events on the launching stream, steps launched asynchronously, barrier + "
                                 "synchronise either side, max over ranks; Python's cyclic GC paused for the K steps",
                       "api": api.name + ": (df * b + c)._query_compiler.execute()"},
            "checked": map_checked, "parity_ok": parity_ok, "parity_failed": parity_fails,
            "roofline": roofline, "roofline_groupby": roofline_groupby, "cpu_baseline": cpu,
            "e2e": e2e, "e2e_groupby": e2e_groupby, "gpu_launches": launches_timed,
            "clocks": clocks, "also": also,
        }  # fmt: skip
        print(json.dumps(line), flush=True)
    if distributed:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
