"""GPU parity of the Fold and Reduce templates (``-m gpu``): the cumulative-function kernels of csrc/cum.cu through the
C ABI (``mb200_cum_partials`` / ``mb200_cum_carry`` / ``mb200_cum_apply``) and through both front doors, and the
Reduce-registered var / std.

Reference = pandas on the same host rows (``DataFrame.cumsum / cummax / cummin / ffill``; the reference's Fold runs
exactly those on the gathered column partition, qc.py:2429-2431, 2809-2810).  Bar: max / min / forward fill and every
int64 result bit for bit; float running sums within ``4 log2(n) 2^-53 * running sum of |x|`` (the tile tree
re-associates pandas' sequential loop); NaN positions identical.  Sizes straddle the 4096-row tile (0, 1, 4095, 4096,
4097), cross many tiles, use views that are only 8-byte aligned, and split one column into three
"ranks" whose carries come from ``mb200_cum_carry`` -- the multi-GPU path without a second GPU.
"""

import math
import os

import numpy as np
import pandas
import pytest

from modin_b200 import synth

pytestmark = pytest.mark.gpu

EPS = 2.0**-53
PANDAS = {"sum": "cumsum", "max": "cummax", "min": "cummin", "ffill": "ffill"}


def _cols(arrays):
    from modin_b200.block import DeviceColumn

    return [DeviceColumn.from_numpy(np.ascontiguousarray(a)) for a in arrays]


def _check(op, got, x):
    want = getattr(pandas.Series(x), PANDAS[op])().to_numpy()
    assert got.dtype == want.dtype and got.shape == want.shape
    if op == "sum" and x.dtype == np.float64:
        assert np.array_equal(np.isnan(got), np.isnan(want))
        bound = 4.0 * max(1.0, math.log2(max(len(x), 2))) * EPS * np.cumsum(np.abs(np.nan_to_num(x))) + 1e-300
        ok = np.isnan(want) | (np.abs(got - want) <= bound)
        assert ok.all(), (op, len(x), int((~ok).sum()))
    else:
        assert np.array_equal(got, want, equal_nan=True), (op, len(x))


def _host_columns(n, seed):
    rng = np.random.RandomState(seed)
    f = rng.randn(n)
    f[rng.rand(n) < 0.15] = np.nan
    if n > 8:
        f[:3] = np.nan  # nothing valid yet at the top
        f[n // 2 : n // 2 + 5] = np.nan
    g = rng.randn(n)  # no NaN at all
    i = rng.randint(-(1 << 40), 1 << 40, size=n).astype(np.int64)
    return f, g, i


@pytest.mark.parametrize("n", [0, 1, 2, 4095, 4096, 4097, 8192, 100_003, (1 << 21) + 5])
def test_cumulative_kernels_against_pandas(n):
    from modin_b200 import ops

    f, g, i = _host_columns(n, seed=n % 97)
    for op in ("sum", "max", "min", "ffill"):
        host = [f, g] if op == "ffill" else [f, g, i]  # float and int columns in one call: one launch group per dtype
        cols = _cols(host)
        state = ops.cum_partials(op, cols)
        outs = ops.cum_apply(state, cols)
        for x, o in zip(host, outs):
            _check(op, o.to_numpy(), x)
        # the column totals the ranks would exchange
        for (code, idxs, _s, totals) in state.groups:
            tot = totals.cpu().numpy()
            for pos, j in enumerate(idxs):
                x = host[j]
                v = x[~np.isnan(x)] if x.dtype == np.float64 else x
                if len(v) == 0:
                    continue
                if op == "sum":
                    assert abs(tot[pos] - v.sum()) <= 4.0 * max(1.0, math.log2(max(n, 2))) * EPS * np.abs(v).sum() + 1e-300
                else:
                    assert tot[pos] == {"max": v.max, "min": v.min, "ffill": lambda: v[-1]}[op]()


def test_cumulative_on_unaligned_views_and_many_columns():
    """Columns that start 8 bytes into an allocation (row slices of a block) and more than 32 columns per call."""
    from modin_b200 import ops
    from modin_b200.block import DeviceColumn

    n = 50_001
    rng = np.random.RandomState(5)
    base = [rng.randn(n + 1) for _ in range(35)]
    for b in base[::3]:
        b[rng.rand(n + 1) < 0.1] = np.nan
    views = []
    for b in base:
        c = DeviceColumn.from_numpy(b)
        views.append(DeviceColumn(c.data[1:], np.float64))  # 8-byte aligned only
    for op in ("sum", "ffill"):
        state = ops.cum_partials(op, views)
        outs = ops.cum_apply(state, views)
        for b, o in zip(base, outs):
            _check(op, o.to_numpy(), b[1:])


@pytest.mark.parametrize("op", ["sum", "max", "min", "ffill"])
def test_carries_across_three_shards(op):
    """One column cut into three row shards, scanned shard by shard with the carry ``mb200_cum_carry`` builds from the
    all-gathered totals: the multi-rank path of DevCumulative (functors.py) on one GPU.  A shard with nothing valid
    and NaN runs across the cuts included."""
    from modin_b200 import ops

    t = ops.torch_mod()
    n = 30_011
    rng = np.random.RandomState(9)
    f = rng.randn(n)
    f[rng.rand(n) < 0.2] = np.nan
    f[9_990:10_020] = np.nan  # across the first cut
    g = rng.randn(n)
    g[10_000:20_000] = np.nan  # the whole middle shard
    i = rng.randint(-1000, 1000, size=n).astype(np.int64)
    host = [f, g] if op == "ffill" else [f, g, i]
    cuts = [(0, 10_000), (10_000, 20_000), (20_000, n)]
    shards = [_cols([x[lo:hi] for x in host]) for lo, hi in cuts]
    states = [ops.cum_partials(op, s) for s in shards]
    # what an all_gather of the per-rank totals produces: rank-major [nranks * ncols] per dtype group
    gathered = [t.cat([st.groups[k][3] for st in states]) for k in range(len(states[0].groups))]
    pieces = [[] for _ in host]
    for r, (st, cols) in enumerate(zip(states, shards)):
        carries = ops.cum_carry(st, gathered, r)
        for j, o in enumerate(ops.cum_apply(st, cols, carries)):
            pieces[j].append(o.to_numpy())
    for x, p in zip(host, pieces):
        _check(op, np.concatenate(p), x)


def _front_door_checks(pd_mod, real_modin):
    pdf = synth.host_frame(200_003, 3, seed=4, nan_per_64k=4000, key_modulus=1000)
    df = pd_mod.DataFrame(pdf)
    fcols = ["c0", "c1", "c2"]
    if real_modin:
        calls = {"cumsum": lambda d: d.cumsum(), "cummax": lambda d: d.cummax(), "cummin": lambda d: d.cummin(),
                 "ffill": lambda d: d.ffill()}  # fmt: skip
        to_pandas = lambda r: r._to_pandas()  # noqa: E731
    else:  # the mirror's API layer is frozen: the templates are reached through its query compiler
        calls = {"cumsum": lambda d: d._query_compiler.cumsum(0), "cummax": lambda d: d._query_compiler.cummax(0),
                 "cummin": lambda d: d._query_compiler.cummin(0), "ffill": lambda d: d._query_compiler.fillna(method="ffill")}  # fmt: skip
        to_pandas = lambda r: r.to_pandas()  # noqa: E731
    for name, call in calls.items():
        got, want = to_pandas(call(df[fcols])), getattr(pdf[fcols], name)()
        assert got.index.equals(want.index) and list(got.columns) == fcols
        for c in fcols:
            _check({"cumsum": "sum", "cummax": "max", "cummin": "min", "ffill": "ffill"}[name], got[c].to_numpy(),
                   pdf[c].to_numpy())  # fmt: skip
    got = to_pandas(calls["cumsum"](df[["key"]]))
    assert got["key"].to_numpy().dtype == np.int64 and np.array_equal(got["key"].to_numpy(), pdf["key"].cumsum().to_numpy())
    # Reduce template: var / std as one device functor per column partition
    if real_modin:
        for name in ("var", "std"):
            for ddof in (1, 0):
                got, want = getattr(df[fcols], name)(ddof=ddof)._to_pandas(), getattr(pdf[fcols], name)(ddof=ddof)
                assert list(got.index) == fcols and np.allclose(got.to_numpy(), want.to_numpy(), rtol=1e-12, atol=0)
    else:
        got, want = df[fcols]._query_compiler.var(), pdf[fcols].var()
        assert np.allclose(got.to_numpy(), want.to_numpy(), rtol=1e-12, atol=0)


def test_fold_and_reduce_through_the_mirror():
    import modin_b200.pandas as bpd

    _front_door_checks(bpd, False)


def test_fold_and_reduce_through_real_modin():
    from tests.test_alignment_merge import REF, _modin

    if not os.path.isdir(os.path.join(REF, "modin")):
        pytest.skip("oracle/_ref (the unmodified reference) is not installed on this box")
    _front_door_checks(_modin(nparts=1), True)


def test_cumulative_over_many_tiles():
    """2^25 rows x 4 float64 generated on the device (8192 tiles per column, so the per-column scan of the tile
    aggregates runs 8 tiles per thread): running sum and running max of two columns against pandas on the host copy."""
    from modin_b200 import ops

    n = 1 << 25
    df = synth.device_frame(n, 4, seed=7, nan_per_64k=500)
    blk = df._query_compiler._modin_frame._partitions[0, 0].get()
    cols = list(blk.cols)
    for op in ("sum", "max"):
        state = ops.cum_partials(op, cols)
        outs = ops.cum_apply(state, cols)
        for c, o in zip(cols[:2], outs[:2]):
            _check(op, o.to_numpy(), c.to_numpy())
