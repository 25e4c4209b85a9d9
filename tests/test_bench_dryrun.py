"""``bench.py``'s GPU arm, dry-run on the numpy device double under gloo (tests/bench_dryrun.py): every rank must
reach every collective at the world sizes the driver runs (a leg only some ranks enter is a hang on the real box --
round 2 found one at 8 ranks this way: a rank whose shard a filter had emptied left Modin's device path), the JSON
line must be well formed and every ``checked`` / ``parity_ok`` true.  Nothing is measured."""

import json
import math
import os
import socket
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _dry_run(ws, extra=()):
    """tests/bench_dryrun.py at world size `ws`; the JSON line rank 0 printed."""
    script = os.path.join(ROOT, "tests", "bench_dryrun.py")
    args = ["--rows", "400000", "--groups", "5000", "--steps", "3", "--warmup", "1", "--e2e-rows", "80000", *extra]
    env = dict(os.environ, MB200_DRYRUN_HANG_DUMP_S="240")
    if ws == 1:
        cmd = [sys.executable, script] + args
    else:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={ws}", "--master-addr",
               "127.0.0.1", "--master-port", str(_free_port()), script, "--gpus", str(ws)] + args  # fmt: skip
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=420, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, "rank 0 prints exactly one JSON line"
    return json.loads(lines[0])


@pytest.mark.parametrize("ws", [1, 2, 8])
def test_bench_control_flow_on_the_double(ws):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: the real bench runs")
    j = _dry_run(ws)
    assert j["n_gpus"] == ws and j["checked"] is True
    assert j["parity_ok"] is (True if ws > 1 else None), j.get("parity_failed")
    legs = j["also"]
    assert len(legs) == 9 and all(a.get("checked") is True for a in legs), [(a["metric"][:40], a.get("checked"), a.get("error")) for a in legs]
    assert j["roofline_groupby"]["checked"] is True
    assert j["e2e"]["checked"] is True and j["e2e_groupby"]["checked"] is True
    for key in ("metric", "value", "unit", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "data",
                "config", "roofline", "e2e", "gpu_launches", "clocks"):  # fmt: skip
        assert key in j, key
    assert "modin.pandas" in j["config"]["api"] or not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "modin"))


DUMPED = [*(f"{leg}{part}" for leg in ("map_abc", "map_fma3", "fold_cumsum", "merge_left_dense", "merge_left_hash")
            for part in ("", "_rows")),
          *(f"{leg}{part}" for leg in ("groupby_sum_dense", "groupby_sum_hash", "groupby_sum_skewed", "e2e_map_abc",
                                       "e2e_groupby_sum") for part in ("", "_index")),
          "reduce_sum", "reduce_mean"]  # fmt: skip


def test_bench_dump_outputs_on_the_double(tmp_path):
    """``--dump-outputs`` at two ranks (the groupby dump gathers over the ranks, so every rank must take part): every
    leg's file is written, in float64 and within 64 MB, and a second run with the same arguments writes the same
    values -- groupby sums within the sum tolerance, everything else bit for bit."""
    import numpy as np
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: the real bench runs")
    dirs = [tmp_path / "a", tmp_path / "b"]
    for d in dirs:
        j = _dry_run(2, ["--dump-outputs", str(d)])
        assert j["checked"] is True and all(a.get("checked") is True for a in j["also"])
    names = sorted(p.name[:-4] for p in dirs[0].iterdir())
    assert names == sorted(DUMPED)
    assert sum(p.stat().st_size for p in dirs[0].iterdir()) <= 64 << 20
    for name in names:
        a, b = (np.load(d / f"{name}.npy") for d in dirs)
        assert a.dtype == np.float64 and a.shape == b.shape and a.size > 0, name
        if name.startswith(("groupby_sum", "e2e_groupby_sum")) and not name.endswith("_index"):
            # the sum tolerance 4 log2(n) 2^-53 sum|x| for n = 400000 rows in one group, every |x| < 8 (synth.gen_f64)
            tol = 4.0 * math.log2(400_000) * 2.0**-53 * 400_000 * 8
            assert np.allclose(a, b, rtol=0, atol=tol, equal_nan=True), name
        else:
            assert ((a == b) | (np.isnan(a) & np.isnan(b))).all(), name
    rows = np.load(dirs[0] / "map_abc_rows.npy")
    assert rows[0] == 0 and (np.diff(rows) > 0).all()
