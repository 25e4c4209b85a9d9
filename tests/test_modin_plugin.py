"""The drop-in boundary under REAL Modin: ``modin_b200.modin_plugin.register()`` plugs the execution
in behind ``modin.pandas`` and the hot-path operations run through Modin's own API layer, query
compiler caster, operator templates and ``PandasDataframe`` methods into this package's partition
classes and device functors.

Modin comes from ``oracle/_ref`` (installed by ``build()`` from the original project, git-ignored; it
travels to the GPU box with the snapshot).  Without it these tests are skipped.  On a box without a
GPU the device is the numpy test double (host logic only); the ``gpu``-marked variant at the bottom
runs the same scenarios on the B200.
"""

import os
import sys

import numpy as np
import pandas
import pytest

from modin_b200 import synth
from oracle import reference_path as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")

pytestmark = pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "modin")),
                                reason="reference Modin not installed under oracle/_ref")  # fmt: skip


def _same(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and bool(((a == b) | (np.isnan(a) & np.isnan(b))).all())


@pytest.fixture(scope="module")
def modin_b200_execution():
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import warnings

    warnings.filterwarnings("ignore")
    from modin_b200 import modin_plugin

    ns = modin_plugin.register()
    import modin
    import modin.config as cfg
    import modin.pandas as mpd

    modin.set_execution(engine="B200", storage_format="Arrow")
    cfg.NPartitions.put(4)
    from modin_b200 import config

    old = config.NPartitions.get()
    config.NPartitions.put(4)
    yield ns, mpd
    config.NPartitions.put(old)


def _scenarios(mpd, ns):
    pdf = synth.host_frame(2003, 4, seed=11, nan_per_64k=3000, key_modulus=23)
    vals = pdf.drop(columns="key")
    mdf = mpd.DataFrame(vals)
    qc = mdf._query_compiler
    assert type(qc) is ns.QueryCompiler and type(qc._modin_frame) is ns.Dataframe
    assert qc.engine == "B200" and qc.storage_format == "Arrow" and qc.get_backend() == "B200"
    from modin_b200.block import DeviceBlock

    assert all(isinstance(p.get(), DeviceBlock) for p in qc._modin_frame._partitions.flatten())
    P = lambda x: x._to_pandas()  # noqa: E731

    assert _same(P(mdf.abs()).to_numpy(), orc.df_abs(vals, 4).to_numpy())
    assert _same(P(mdf * 1.5 + 0.25).to_numpy(), orc.a_mul_b_add_c(vals, 1.5, 0.25, 4).to_numpy())
    assert _same(P(-mdf).to_numpy(), (-vals).to_numpy())
    assert _same(P(mdf.isna()).to_numpy().astype(float), vals.isna().to_numpy().astype(float))
    assert _same(P(mdf.fillna(2.0)).to_numpy(), orc.df_fillna(vals, 2.0, 4).to_numpy())
    assert _same(P(mdf.round(2)).to_numpy(), orc.df_round(vals, 2, 4).to_numpy())
    assert _same(P(mdf.clip(-0.5, 0.75)).to_numpy(), orc.df_clip(vals, -0.5, 0.75, 4).to_numpy())
    assert np.allclose(P(mdf.prod()).to_numpy(), orc.df_prod(vals, 4).to_numpy(), rtol=1e-9, atol=0, equal_nan=True)
    mask, pmask = (mdf > 0.0) & (mdf < 1.0), (vals > 0.0) & (vals < 1.0)
    assert _same(P(mask).to_numpy().astype(float), pmask.to_numpy().astype(float))
    assert _same(P(~mask | (mdf > 2.0)).to_numpy().astype(float), (~pmask | (vals > 2.0)).to_numpy().astype(float))
    assert list(P(mask.sum()).to_numpy()) == list(pmask.sum().to_numpy())
    assert list(P(mask.any()).to_numpy()) == list(pmask.any().to_numpy())
    assert list(P((mdf > -100.0).all()).to_numpy()) == list((vals > -100.0).all().to_numpy())
    other = synth.host_frame(2003, 4, seed=12)
    mo = mpd.DataFrame(other)
    assert _same(P(mdf * mo + mo).to_numpy(), orc.a_mul_b_add_c(vals, other, other, 4).to_numpy())
    assert _same(P(mdf < mo).to_numpy().astype(float), (vals < other).to_numpy().astype(float))

    s = P(mdf.sum())
    assert isinstance(s, pandas.Series) and list(s.index) == list(vals.columns)
    assert np.allclose(s.to_numpy(), orc.df_sum(vals, 4).to_numpy(), rtol=0, atol=1e-9)
    assert np.allclose(P(mdf.mean()).to_numpy(), orc.df_mean(vals, 4).to_numpy(), rtol=0, atol=1e-12)
    assert _same(P(mdf.count()).to_numpy(), orc.df_count(vals, 4).to_numpy())
    assert _same(P(mdf.min()).to_numpy(), orc.df_min(vals, 4).to_numpy())
    assert _same(P(mdf.max()).to_numpy(), orc.df_max(vals, 4).to_numpy())

    mfull = mpd.DataFrame(pdf)
    g = P(mfull.groupby("key").sum())
    want = orc.groupby_reduce(pdf, "key", "sum", 4)
    assert list(g.index) == list(want.index) and list(g.columns) == list(want.columns)
    assert np.allclose(g.to_numpy(), want.to_numpy(), rtol=0, atol=1e-9)
    assert _same(P(mfull.groupby("key").count()).to_numpy(), orc.groupby_reduce(pdf, "key", "count", 4).to_numpy())
    assert np.allclose(P(mfull.groupby("key").mean()).to_numpy(), orc.groupby_reduce(pdf, "key", "mean", 4).to_numpy(),
                       rtol=0, atol=1e-12, equal_nan=True)  # fmt: skip

    rng = np.random.RandomState(1)
    dim = pandas.DataFrame({"key": rng.permutation(23)[:20].astype(np.int64), "d0": rng.randn(20)})
    left = P(mfull.merge(mpd.DataFrame(dim), on="key", how="left"))
    wl = orc.broadcast_merge(pdf, dim, "key", "left", 4)
    assert list(left.columns) == list(wl.columns) and _same(left.to_numpy(), wl.to_numpy())
    inner = P(mfull.merge(mpd.DataFrame(dim), on="key", how="inner"))
    assert _same(inner.to_numpy(), orc.broadcast_merge(pdf, dim, "key", "inner", 4).to_numpy())


def _late_scenarios(mpd, ns):
    """astype / drop_duplicates / Series.unique / concat / nunique through real ``modin.pandas``.  Kept apart from
    ``_scenarios``: these were added after the round's GPU minutes were spent, so their GPU variant lives in the
    late-sorting tests/test_zz_gpu_row_selection.py and cannot hide the hardware-verified scenarios behind ``-x``.
    ``equals`` compares values, row labels, column labels and dtypes."""
    pdf = synth.host_frame(2003, 3, seed=11, nan_per_64k=3000, key_modulus=23)
    pb = synth.host_frame(1001, 3, seed=12, nan_per_64k=3000, key_modulus=23)
    pdf["k2"], pb["k2"] = synth.gen_i64(2003, 98, 1, 7) * 5 - 10, synth.gen_i64(1001, 97, 1, 7) * 5 - 10
    mdf, mb = mpd.DataFrame(pdf), mpd.DataFrame(pb)
    assert type(mdf._query_compiler) is ns.QueryCompiler
    P = lambda x: x._to_pandas()  # noqa: E731

    assert P(mdf.astype("float64")).equals(pdf.astype("float64"))
    assert P(mdf.astype({"key": "float64"})).equals(pdf.astype({"key": "float64"}))
    with pytest.raises(NotImplementedError):
        mdf.astype("int64")  # float64 -> int64 truncation is not on the path; refused before any launch
    for keep in ("first", "last"):
        for ignore in (False, True):
            got = P(mdf.drop_duplicates(subset=["key"], keep=keep, ignore_index=ignore))
            assert got.equals(pdf.drop_duplicates(subset=["key"], keep=keep, ignore_index=ignore)), (keep, ignore)
    assert P(mdf.drop_duplicates(subset="k2")).equals(pdf.drop_duplicates(subset="k2"))
    assert np.array_equal(mdf["key"].unique(), pdf["key"].unique())  # values in order of first appearance
    assert P(mdf["k2"].drop_duplicates()).equals(pdf["k2"].drop_duplicates())
    with pytest.raises(NotImplementedError):
        mdf.drop_duplicates()  # all columns
    with pytest.raises(NotImplementedError):
        mdf.drop_duplicates(subset=["key"], keep=False)
    with pytest.raises(KeyError):
        mdf.drop_duplicates(subset=["nope"])
    for ignore in (False, True):
        assert P(mpd.concat([mdf, mb, mdf], ignore_index=ignore)).equals(pandas.concat([pdf, pb, pdf], ignore_index=ignore))
    cat, wcat = mpd.concat([mdf, mb], ignore_index=True), pandas.concat([pdf, pb], ignore_index=True)
    assert _same(P(cat * 2.0).to_numpy(), (wcat * 2.0).to_numpy())
    fl = ["key", "c0", "c1", "c2"]  # device groupby.sum aggregates float64 value columns only
    g, wg = P(cat[fl].groupby("key").sum()), wcat[fl].groupby("key").sum()
    assert list(g.index) == list(wg.index) and np.allclose(g.to_numpy(), wg.to_numpy(), rtol=0, atol=1e-9)
    assert P(mdf[["key", "k2"]].nunique()).equals(pdf[["key", "k2"]].nunique())
    assert mdf["key"].nunique() == pdf["key"].nunique()
    with pytest.raises(NotImplementedError):
        mdf.nunique()  # float columns
    with pytest.raises(NotImplementedError):
        mdf.reset_index()  # labels -> column is not on the path; drop=True is
    dd, wdd = mdf.drop_duplicates(subset=["key"], keep="last"), pdf.drop_duplicates(subset=["key"], keep="last")
    assert P(dd.reset_index(drop=True)).equals(wdd.reset_index(drop=True))  # non-range labels -> 0..K-1

    # Series comparisons (qc.series_gt ...), logical ops between Series, and what hangs off them
    assert P(mdf["c0"] > 0.0).equals(pdf["c0"] > 0.0) and P(mdf["key"] == 3).equals(pdf["key"] == 3)
    assert P(mdf["c0"] >= mdf["c1"]).equals(pdf["c0"] >= pdf["c1"])
    assert P((mdf["c0"] > 0.0) & (mdf["c1"] < 0.0)).equals((pdf["c0"] > 0.0) & (pdf["c1"] < 0.0))
    assert P(mdf[mdf["c0"] > 0.5]).equals(pdf[pdf["c0"] > 0.5])  # boolean row selection, labels kept
    assert P(mdf[(mdf["c0"] > 0.0) | (mdf["key"] == 3)]).equals(pdf[(pdf["c0"] > 0.0) | (pdf["key"] == 3)])
    assert P(mdf[mdf["c0"] > 100.0]).shape == (0, pdf.shape[1])
    sel, wsel = mdf[mdf["c0"] > 0.0], pdf[pdf["c0"] > 0.0]
    assert np.allclose(P(sel[["c0", "c1", "c2"]].sum()).to_numpy(), wsel[["c0", "c1", "c2"]].sum().to_numpy(), rtol=0, atol=1e-9)
    assert P(mdf.dropna()).equals(pdf.dropna())
    assert P(mdf.dropna(how="all", subset=["c0", "c1"])).equals(pdf.dropna(how="all", subset=["c0", "c1"]))
    with pytest.raises(NotImplementedError):
        mdf.dropna(axis=1)
    assert P(mdf[["key", "k2"]].isin([3, 7, -10, 20])).equals(pdf[["key", "k2"]].isin([3, 7, -10, 20]))
    assert P(mdf[mdf["key"].isin([1, 2, 3])]).equals(pdf[pdf["key"].isin([1, 2, 3])])
    assert P(mdf.assign(d=mdf["c0"] * 2.0)).equals(pdf.assign(d=pdf["c0"] * 2.0))
    assert P(mdf.head(7)).equals(pdf.head(7))
    # var / std: a different summation order than pandas, so the last bits may differ (rtol, not equals)
    fcols = ["c0", "c1", "c2"]
    for ddof in (1, 0):
        got, want = P(mdf[fcols].var(ddof=ddof)), pdf[fcols].var(ddof=ddof)
        assert list(got.index) == list(want.index) and np.allclose(got.to_numpy(), want.to_numpy(), rtol=1e-12, atol=0)
    assert np.allclose(P(mdf[fcols].std()).to_numpy(), pdf[fcols].std().to_numpy(), rtol=1e-12, atol=0)
    with pytest.raises(NotImplementedError):
        mdf[fcols].var(axis=1)
    # Binary template operand shapes through Modin's own dispatch: reflected scalars, positional / labelled row vectors
    # (Modin applies those full-axis), a column along axis 0 (its broadcast branch squeezes the one-column block),
    # co-partitioned frames, a frame-valued fillna
    v, other = pdf[fcols], synth.host_frame(2003, 3, seed=13, nan_per_64k=2000)[fcols]
    dv, do = mdf[fcols], mpd.DataFrame(other)
    row3, srow = [0.5, -1.0, 2.0], pandas.Series([0.5, -1.0, 2.0], index=fcols)
    for name, got, want in (
        ("2 - df", 2.0 - dv, 2.0 - v), ("1 / df", 1.0 / dv, 1.0 / v), ("df.rsub", dv.rsub(1.0), v.rsub(1.0)),
        ("df + list", dv + row3, v + row3), ("df * Series", dv * srow, v * srow), ("df < list", dv < row3, v < row3),
        ("df.mul(col, 0)", dv.mul(dv["c1"], axis=0), v.mul(v["c1"], axis=0)),
        ("df.rsub(col, 0)", dv.rsub(dv["c1"], axis=0), v.rsub(v["c1"], axis=0)),
        ("df.lt(col, 0)", dv.lt(dv["c1"], axis=0), v.lt(v["c1"], axis=0)),
        ("df - other", dv - do, v - other), ("df.rtruediv(other)", dv.rtruediv(do), v.rtruediv(other)),
        ("a*b+c", dv * do + do, v * other + other), ("a*list+list", dv * row3 + row3, v * row3 + row3),
        ("fillna(frame)", dv.fillna(do), v.fillna(other)), ("fillna(dict)", dv.fillna({"c0": 1.0}), v.fillna({"c0": 1.0})),
        ("series - series", dv["c0"] - dv["c1"], v["c0"] - v["c1"]), ("2 - series", 2.0 - dv["c0"], 2.0 - v["c0"]),
    ):  # fmt: skip
        assert P(got).equals(want), name
    # sort_values: stable, NaN last (the reference's own range-partitioning sort returns an empty frame under pandas 3)
    for by, asc in (("c0", True), ("c0", False), ("key", True), ("k2", False)):
        assert P(mdf.sort_values(by, ascending=asc)).equals(pdf.sort_values(by, ascending=asc, kind="stable")), (by, asc)
    assert P(mdf.sort_values("c1", ignore_index=True)).equals(pdf.sort_values("c1", kind="stable", ignore_index=True))
    sel, wsel = mdf[mdf["c0"] > 0.0], pdf[pdf["c0"] > 0.0]
    assert P(sel.sort_values("c2")).equals(wsel.sort_values("c2", kind="stable"))  # labels ride along as a device column
    assert P(mdf.sort_values("c0").head(10)).equals(pdf.sort_values("c0", kind="stable").head(10))
    with pytest.raises(NotImplementedError):
        mdf.sort_values(["c0", "c1"])
    with pytest.raises(NotImplementedError):
        mdf.sort_values("c0", na_position="first")
    with pytest.raises(KeyError):
        mdf.sort_values("nope")
    # a query-compiler method the plug-in does not override reaches the blocks with Modin's pandas lambda: refused
    # with a message that says so (it used to be a bare AttributeError on the block)
    with pytest.raises(NotImplementedError, match="no device implementation"):
        P(mdf[fcols].median())
    # Fold template (alg/fold.py): cumulative functions and forward fill down the rows, NaN skipped like pandas does
    got, want = P(mdf[fcols].cumsum()), pdf[fcols].cumsum()
    assert got.index.equals(want.index) and np.allclose(got.to_numpy(), want.to_numpy(), rtol=0, atol=1e-9, equal_nan=True)
    assert np.array_equal(np.isnan(got.to_numpy()), np.isnan(want.to_numpy()))
    assert P(mdf[fcols].cummax()).equals(pdf[fcols].cummax()) and P(mdf[fcols].cummin()).equals(pdf[fcols].cummin())
    assert P(mdf[["key", "k2"]].cumsum()).equals(pdf[["key", "k2"]].cumsum())  # int64: exact
    assert P(mdf["c1"].cummax()).equals(pdf["c1"].cummax())
    assert P(mdf.ffill()).equals(pdf.ffill())
    with pytest.raises(NotImplementedError):
        mdf[fcols].cumsum(skipna=False)
    with pytest.raises(NotImplementedError):
        mdf.ffill(limit=2)


def test_odd_shapes_under_real_modin_cpu_double(modin_b200_execution, cpu_device):
    """Wide frames (two column partitions), empty results, frames whose labels are device index columns (filter /
    groupby results) through real ``modin.pandas`` with the plug-in: values, row labels, column labels vs pandas."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: host-logic sweep, runs on the double only")
    ns, mpd = modin_b200_execution
    rng = np.random.RandomState(7)
    W = 40
    fcols = [f"w{i}" for i in range(W)]
    wide = pandas.DataFrame(rng.randn(300, W), columns=fcols)
    wide.iloc[::17, 3] = np.nan
    wide.iloc[::29, 35] = np.nan
    wide.insert(0, "key", rng.randint(0, 7, 300).astype(np.int64))
    pa = synth.host_frame(1003, 3, seed=1, nan_per_64k=3000, key_modulus=11)
    dim = pandas.DataFrame({"key": rng.permutation(11)[:9].astype(np.int64), "d0": rng.randn(9)})
    dw, a, dd = mpd.DataFrame(wide), mpd.DataFrame(pa), mpd.DataFrame(dim)
    assert dw._query_compiler._modin_frame._partitions.shape[1] == 2
    f = ["c0", "c1", "c2"]
    emp, wemp = a[a["c0"] > 100.0], pa[pa["c0"] > 100.0]
    fl, wfl = a[a["c0"] > 0.0], pa[pa["c0"] > 0.0]
    g, wg = a.groupby("key").sum(), pa.groupby("key").sum()
    cases = {
        "wide": (lambda: dw, lambda: wide),
        "wide filter": (lambda: dw[dw["w0"] > 0.0], lambda: wide[wide["w0"] > 0.0]),
        "wide dropna": (lambda: dw.dropna(), lambda: wide.dropna()),
        "wide astype": (lambda: dw.astype({"key": "float64"}), lambda: wide.astype({"key": "float64"})),
        "wide sum": (lambda: dw[fcols].sum(), lambda: wide[fcols].sum()),
        "wide a*b+c": (lambda: dw[fcols] * dw[fcols] + dw[fcols], lambda: wide[fcols] * wide[fcols] + wide[fcols]),
        "wide comparison": (lambda: dw[fcols] < 0.0, lambda: wide[fcols] < 0.0),
        "wide groupby": (lambda: dw.groupby("key").sum(), lambda: wide.groupby("key").sum()),
        "wide merge": (lambda: dw.merge(dd, on="key", how="left"), lambda: wide.merge(dim, on="key", how="left")),
        "wide concat": (lambda: mpd.concat([dw, dw]), lambda: pandas.concat([wide, wide])),
        "wide head": (lambda: dw.head(77), lambda: wide.head(77)),
        "wide assign": (lambda: dw.assign(z=dw["w1"] * 2.0), lambda: wide.assign(z=wide["w1"] * 2.0)),
        "wide isin": (lambda: dw[["key"]].isin([1, 2]), lambda: wide[["key"]].isin([1, 2])),
        "empty": (lambda: emp, lambda: wemp),
        "empty abs": (lambda: emp[f].abs(), lambda: wemp[f].abs()),
        "empty drop_duplicates": (lambda: emp.drop_duplicates(subset=["key"]), lambda: wemp.drop_duplicates(subset=["key"])),
        "empty astype": (lambda: emp.astype({"key": "float64"}), lambda: wemp.astype({"key": "float64"})),
        "concat with an empty frame": (lambda: mpd.concat([a, emp]), lambda: pandas.concat([pa, wemp])),
        "filter twice": (lambda: fl[fl["c1"] > 0.0], lambda: wfl[wfl["c1"] > 0.0]),
        "filter -> sum": (lambda: fl[f].sum(), lambda: wfl[f].sum()),
        "filter -> groupby": (lambda: fl.groupby("key").mean(), lambda: wfl.groupby("key").mean()),
        "filter -> merge": (lambda: fl.merge(dd, on="key", how="inner"), lambda: wfl.merge(dim, on="key", how="inner")),
        "filter -> square": (lambda: fl[["c0"]] * fl[["c0"]], lambda: wfl[["c0"]] * wfl[["c0"]]),
        "filter -> assign": (lambda: fl.assign(z=fl["c0"] + 1.0), lambda: wfl.assign(z=wfl["c0"] + 1.0)),
        "filter -> drop_duplicates": (lambda: fl.drop_duplicates(subset=["key"], keep="last"),
                                      lambda: wfl.drop_duplicates(subset=["key"], keep="last")),
        "filter -> head": (lambda: fl.head(13), lambda: wfl.head(13)),
        "filter -> tail": (lambda: fl.tail(13), lambda: wfl.tail(13)),
        "filter -> dropna": (lambda: fl.dropna(), lambda: wfl.dropna()),
        "concat of filtered and plain": (lambda: mpd.concat([fl, a]), lambda: pandas.concat([wfl, pa])),
        "group table * 2": (lambda: g * 2.0, lambda: wg * 2.0),
        "group table filter": (lambda: g[g["c0"] > 0.0], lambda: wg[wg["c0"] > 0.0]),
        "group table sum": (lambda: g.sum(), lambda: wg.sum()),
        "group table + itself": (lambda: g + g, lambda: wg + wg),
        "group table head": (lambda: g.head(3), lambda: wg.head(3)),
        "int column > float scalar": (lambda: a[a["key"] > 4.5], lambda: pa[pa["key"] > 4.5]),
        "tail": (lambda: a.tail(9), lambda: pa.tail(9)),
    }  # fmt: skip
    bad = {}
    for name, (dev, host) in cases.items():
        got, want = dev()._to_pandas(), host()
        ok = (list(got.index) == list(want.index) and (not hasattr(want, "columns") or list(got.columns) == list(want.columns))
              and got.shape == want.shape
              and np.allclose(np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64), rtol=1e-12, atol=1e-9, equal_nan=True))  # fmt: skip
        if not ok:
            bad[name] = (got.shape, want.shape, list(got.index)[:3], list(want.index)[:3])
    assert not bad, bad
    with pytest.raises(NotImplementedError, match="one column partition"):
        dw.drop_duplicates(subset=["key"])
    # var / std are a device Reduce per column partition, so a frame wider than one partition works
    gv, wv = dw[fcols].var()._to_pandas(), dw[fcols]._to_pandas().var()
    assert list(gv.index) == list(wv.index) and np.allclose(gv.to_numpy(), wv.to_numpy(), rtol=1e-12, atol=0)
    # NOT covered, and not this package's doing: reductions / filters / groupby of an EMPTY frame make Modin's API
    # layer default to pandas, and that path builds ``pandas.Series(..., fastpath=...)`` (modin/pandas/series.py:166),
    # a keyword pandas 3 removed (the reference pins pandas < 2.4)
    with pytest.raises(TypeError, match="fastpath"):
        emp[f].sum()


def _level_scenarios(mpd):
    """``groupby(level=0)`` through real ``modin.pandas``: the row labels are the key (a device label column, or a range
    materialised on the device); written after the round's last GPU run, so kept out of the scenario set whose
    ``gpu``-marked variant has passed on a B200."""
    pdf = synth.host_frame(2003, 3, seed=11, nan_per_64k=3000)
    fcols = ["c0", "c1", "c2"]
    P = lambda x: x._to_pandas()  # noqa: E731
    for idx in (pandas.Index(np.arange(len(pdf)) % 37 - 5, name="lab"), pandas.RangeIndex(len(pdf)),
                pandas.Index(np.round(np.sin(np.arange(len(pdf))) * 4) / 2, name="f")):
        lp = pdf[fcols].set_axis(idx, axis=0)
        ldf = mpd.DataFrame(lp)
        for agg in ("sum", "count", "max", "size"):
            got, want = P(getattr(ldf.groupby(level=0), agg)()), getattr(lp.groupby(level=0), agg)()
            assert np.array_equal(got.index.to_numpy(), want.index.to_numpy()) and got.index.name == want.index.name, (idx.name, agg)
            assert np.allclose(np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64), rtol=0, atol=1e-9, equal_nan=True)
    assert P(ldf.groupby(level="f").sum()).index.name == "f"
    with pytest.raises(ValueError, match="only valid with MultiIndex"):
        ldf.groupby(level=1).sum()
    with pytest.raises(ValueError, match="not the name of the index"):
        ldf.groupby(level="nope").sum()


def test_late_additions_under_real_modin_cpu_double(modin_b200_execution, cpu_device):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu-marked test")
    ns, mpd = modin_b200_execution
    _late_scenarios(mpd, ns)
    _level_scenarios(mpd)


def test_late_gpu_plugin_test_is_sound_on_the_double(modin_b200_execution, cpu_device, monkeypatch):
    """The gpu-marked variant of the late scenarios (tests/test_zz_gpu_row_selection.py) has not run on a B200 yet;
    run its body here so that its scaffolding (registration, scenario import) is known to work.  Only the
    kernel-launch counter is stubbed: the double launches nothing, which is exactly what that assertion is there
    to catch on a GPU box."""
    import importlib.util

    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: the real test runs")
    from modin_b200 import _lib

    class _Counter:
        n = 0

        def mb200_launch_count(self):
            _Counter.n += 1
            return _Counter.n

    monkeypatch.setattr(_lib, "load", lambda: _Counter())
    spec = importlib.util.spec_from_file_location("late_gpu_tests", os.path.join(ROOT, "tests", "test_zz_gpu_row_selection.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.test_late_additions_under_real_modin_on_b200()
    assert _Counter.n == 2  # bracketed the scenarios: read once before, once after


def test_registration_resolves_through_modins_dispatcher(modin_b200_execution):
    ns, mpd = modin_b200_execution
    import modin.config as cfg
    from modin.core.execution.dispatching.factories.dispatcher import FactoryDispatcher

    assert cfg.Engine.get() == "B200" and cfg.StorageFormat.get() == "Arrow"
    factory = FactoryDispatcher.get_factory()
    assert factory.io_cls is ns.IO
    assert ns.IO.frame_cls is ns.Dataframe and ns.IO.query_compiler_cls is ns.QueryCompiler


def test_hot_path_under_real_modin_cpu_double(modin_b200_execution, cpu_device):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu-marked test")
    ns, mpd = modin_b200_execution
    _scenarios(mpd, ns)


@pytest.mark.gpu
def test_hot_path_under_real_modin_on_b200(modin_b200_execution):
    ns, mpd = modin_b200_execution
    from modin_b200 import _lib

    lib = _lib.load()
    before = lib.mb200_launch_count()
    _scenarios(mpd, ns)
    assert lib.mb200_launch_count() > before


# ------------------------------------------------------------------------------------------------------------
# The plug-in under torch.distributed (one process per GPU; here 2 gloo ranks on the numpy device double): every
# rank activates the execution, ingests ITS row shard of the same host frame through ``modin.pandas`` and runs the
# hot path; results are compared with whole-frame pandas / the oracle.
def _plugin_rank_job(rank, ws):
    import sys
    import warnings

    warnings.filterwarnings("ignore")
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import cpu_double
    from modin_b200 import config, modin_plugin

    out = {}
    with cpu_double.installed():
        ns = modin_plugin.activate()
        import modin.config as cfg
        import modin.pandas as mpd

        cfg.NPartitions.put(2)
        config.NPartitions.put(2)
        pdf = synth.host_frame(2003, 4, seed=11, nan_per_64k=3000, key_modulus=23)
        vals = pdf.drop(columns="key")
        mdf, mfull = mpd.DataFrame(vals), mpd.DataFrame(pdf)
        fr = mdf._query_compiler._modin_frame
        assert type(fr) is ns.Dataframe
        lo, hi = (rank * 2003) // ws, ((rank + 1) * 2003) // ws  # shard_bounds for an even-ish split
        out["local_rows"] = (len(fr), int(mdf.index[0]), int(mdf.index[-1]))
        out["job_rows"] = len(mdf)  # Modin's API sees the job-wide row count (its emptiness test must agree on all ranks)
        # a filter that leaves some ranks EMPTY must not make them leave the device path (Modin defaults every
        # method of an empty frame to pandas, modin/pandas/base.py:4372): the reduction after it is a collective
        withpos = vals.assign(pos=np.arange(len(vals), dtype=np.float64))
        mpos = mpd.DataFrame(withpos)
        first_rows = mpos[mpos["pos"] < 10.0]  # only rank 0 holds such rows
        out["sum_after_one_sided_filter"] = first_rows.sum()._to_pandas()
        out["len_after_one_sided_filter"] = len(first_rows)
        P = lambda x: x._to_pandas()  # noqa: E731
        lazy = mdf * 1.5 + 0.25
        out["len_of_lazy"] = len(lazy)  # asking for the length must not run the queued ops one by one
        out["queued"] = [len(p.call_queue) for p in lazy._query_compiler._modin_frame._partitions.flatten()]
        out["affine"] = P(mdf * 1.5 + 0.25)
        out["abs"] = P(mdf.abs())
        out["lt"] = P(mdf < 0.0)
        other = mpd.DataFrame(synth.host_frame(2003, 4, seed=12))
        out["fma3"] = P(mdf * other + other)
        out["fillna_frame"] = P(mdf.fillna(other))
        for name in ("sum", "mean", "count", "min", "max", "var", "std"):
            out[name] = P(getattr(mdf, name)())
        g = mfull.groupby("key")
        for agg in ("sum", "count", "mean", "size", "min", "max"):
            r = getattr(g, agg)()
            out["gb_" + agg] = P(r)
            out["gb_local_" + agg] = sum(r._query_compiler._modin_frame.row_lengths)  # this rank's key range
            out["gb_job_" + agg] = len(r)  # len() of a frame is job-wide under torch.distributed
        for name in ("cumsum", "cummax", "cummin", "ffill"):  # Fold: each rank scans its shard, carries cross the ranks
            out[name] = P(getattr(mdf, name)())
        edge = vals.copy()  # NaN runs across the shard boundary (row 1001) and at the very top
        edge.iloc[995:1010, 0] = np.nan
        edge.iloc[0:5, 1] = np.nan
        edge.iloc[1001:, 2] = np.nan  # a shard with nothing valid in one column
        medge = mpd.DataFrame(edge)
        for name in ("cumsum", "cummax", "ffill"):
            out["edge_" + name] = P(getattr(medge, name)())
        fkey = pdf.assign(fk=np.where(np.arange(len(pdf)) % 17 == 0, np.nan, np.round(pdf["c0"].fillna(0.0) * 2.0, 0) / 2.0))
        mfk = mpd.DataFrame(fkey.drop(columns="key"))
        out["gb_float_key"] = P(mfk.groupby("fk").sum())  # the key runs as its int64 image; NaN keys are dropped
        out["gb_float_key_keepna"] = P(mfk.groupby("fk", dropna=False).count())
        out["gb_dict"] = P(g.agg({"c2": "mean", "c0": "sum", "c3": "max"}))  # one device aggregation per function
        rng = np.random.RandomState(1)
        dim = pandas.DataFrame({"key": rng.permutation(23)[:20].astype(np.int64), "d0": rng.randn(20)})
        out["merge_left"] = P(mfull.merge(mpd.DataFrame(dim), on="key", how="left"))
        out["merge_inner"] = P(mfull.merge(mpd.DataFrame(dim), on="key", how="inner"))
        # two key columns: packed into one int64 over the key ranges of both frames, agreed across the ranks
        two = pdf.assign(k2=(np.arange(len(pdf), dtype=np.int64) * 7) % 5 - 2)
        dim2 = pandas.DataFrame({"key": np.repeat(np.arange(23, dtype=np.int64), 5)[:100],
                                 "k2": np.tile(np.arange(-2, 3, dtype=np.int64), 23)[:100], "d1": rng.randn(100)})
        out["merge_two_keys"] = P(mpd.DataFrame(two).merge(mpd.DataFrame(dim2), on=["key", "k2"], how="left"))
        out["filter"] = P(mdf[mdf["c0"] > 0.0])
        out["dropna"] = P(mdf.dropna())
        out["nunique"] = P(mfull[["key"]].nunique())
        out["sort"] = P(mdf.sort_values("c1"))
        # results every rank holds in full (reductions) stay that through maps and further reductions: they must not
        # be combined across the ranks a second time
        out["sum_of_scaled_sums"] = float((mdf.sum() * 2.0).sum())
        out["max_of_means"] = float(mdf.mean().max())
        out["count_positive_sums"] = int((mdf.sum() > 0).sum())
        # equal keys on different ranks: the functor exchanges the keys of the per-rank survivors (sharded result)
        out["dd_last"] = P(mfull.drop_duplicates(subset=["key"], keep="last"))
        out["dd_series"] = P(mfull["key"].drop_duplicates())
        out["dd_then_sum"] = P(mfull.drop_duplicates(subset=["key"])[["c0", "c1"]].sum())  # the result is row-sharded like any frame
    return out


def test_plugin_under_two_gloo_ranks():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: tools/dist_check.py covers the plug-in under NCCL")
    from tests.test_dist_gloo import _run

    outs = _run(_plugin_rank_job, ws=2)
    pdf = synth.host_frame(2003, 4, seed=11, nan_per_64k=3000, key_modulus=23)
    vals = pdf.drop(columns="key")
    other = synth.host_frame(2003, 4, seed=12)
    assert all(o["job_rows"] == 2003 and o["len_of_lazy"] == 2003 for o in outs)
    assert all(q == 2 for o in outs for q in o["queued"]), "x * s + t must still be queued (-> one fused sweep)"
    wpos = vals.assign(pos=np.arange(len(vals), dtype=np.float64))
    for o in outs:
        assert o["len_after_one_sided_filter"] == 10
        assert np.allclose(o["sum_after_one_sided_filter"].to_numpy(), wpos[wpos["pos"] < 10.0].sum().to_numpy(), rtol=0, atol=1e-9)
    rows = [o["local_rows"] for o in outs]
    assert sum(r[0] for r in rows) == 2003 and rows[0][1] == 0 and rows[1][2] == 2002 and rows[0][2] + 1 == rows[1][1]
    rng = np.random.RandomState(1)
    dim = pandas.DataFrame({"key": rng.permutation(23)[:20].astype(np.int64), "d0": rng.randn(20)})
    for o in outs:  # every rank gathers the job-wide result
        assert _same(o["affine"].to_numpy(), orc.a_mul_b_add_c(vals, 1.5, 0.25, 4).to_numpy())
        assert list(o["affine"].index) == list(vals.index)
        assert _same(o["abs"].to_numpy(), vals.abs().to_numpy())
        assert _same(o["lt"].to_numpy().astype(float), (vals < 0.0).to_numpy().astype(float))
        assert _same(o["fma3"].to_numpy(), orc.a_mul_b_add_c(vals, other, other, 4).to_numpy())
        assert _same(o["fillna_frame"].to_numpy(), vals.fillna(other).to_numpy())
        assert np.allclose(o["sum"].to_numpy(), vals.sum().to_numpy(), rtol=0, atol=1e-9)
        assert np.allclose(o["mean"].to_numpy(), vals.mean().to_numpy(), rtol=0, atol=1e-12)
        assert _same(o["count"].to_numpy(), vals.count().to_numpy())
        assert _same(o["min"].to_numpy(), vals.min().to_numpy()) and _same(o["max"].to_numpy(), vals.max().to_numpy())
        assert np.allclose(o["var"].to_numpy(), vals.var().to_numpy(), rtol=1e-12, atol=0)
        assert np.allclose(o["std"].to_numpy(), vals.std().to_numpy(), rtol=1e-12, atol=0)
        for agg in ("sum", "count", "mean", "size", "min", "max"):
            want = orc.groupby_reduce(pdf, "key", agg, 4)
            got = o["gb_" + agg]
            assert list(got.index) == list(want.index), agg
            assert np.allclose(np.asarray(got, dtype=np.float64).reshape(len(want), -1),
                               np.asarray(want, dtype=np.float64).reshape(len(want), -1), rtol=0, atol=1e-9, equal_nan=True), agg  # fmt: skip
        assert np.allclose(o["cumsum"].to_numpy(), vals.cumsum().to_numpy(), rtol=0, atol=1e-9, equal_nan=True)
        assert list(o["cumsum"].index) == list(vals.index)
        for name in ("cummax", "cummin", "ffill"):
            assert o[name].equals(getattr(vals, name)()), name
        edge = vals.copy()
        edge.iloc[995:1010, 0] = np.nan
        edge.iloc[0:5, 1] = np.nan
        edge.iloc[1001:, 2] = np.nan
        assert np.allclose(o["edge_cumsum"].to_numpy(), edge.cumsum().to_numpy(), rtol=0, atol=1e-9, equal_nan=True)
        assert o["edge_cummax"].equals(edge.cummax()) and o["edge_ffill"].equals(edge.ffill())
        fkey = pdf.assign(fk=np.where(np.arange(len(pdf)) % 17 == 0, np.nan, np.round(pdf["c0"].fillna(0.0) * 2.0, 0) / 2.0))
        wfk = fkey.drop(columns="key").groupby("fk").sum()
        assert np.array_equal(o["gb_float_key"].index.to_numpy(), wfk.index.to_numpy())
        assert np.allclose(o["gb_float_key"].to_numpy(), wfk.to_numpy(), rtol=0, atol=1e-9, equal_nan=True)
        wfk = fkey.drop(columns="key").groupby("fk", dropna=False).count()
        assert np.array_equal(o["gb_float_key_keepna"].index.to_numpy(), wfk.index.to_numpy(), equal_nan=True)
        assert np.array_equal(o["gb_float_key_keepna"].to_numpy(), wfk.to_numpy())
        wd_ = pdf.groupby("key").agg({"c2": "mean", "c0": "sum", "c3": "max"})
        assert list(o["gb_dict"].columns) == list(wd_.columns) and list(o["gb_dict"].index) == list(wd_.index)
        assert np.allclose(o["gb_dict"].to_numpy(), wd_.to_numpy(), rtol=0, atol=1e-9, equal_nan=True)
        wl = orc.broadcast_merge(pdf, dim, "key", "left", 4)
        assert list(o["merge_left"].columns) == list(wl.columns) and _same(o["merge_left"].to_numpy(), wl.to_numpy())
        assert _same(o["merge_inner"].to_numpy(), orc.broadcast_merge(pdf, dim, "key", "inner", 4).to_numpy())
        two = pdf.assign(k2=(np.arange(len(pdf), dtype=np.int64) * 7) % 5 - 2)
        rng2 = np.random.RandomState(1)
        rng2.permutation(23), rng2.randn(20)  # the draws the rank job made before building dim2
        dim2 = pandas.DataFrame({"key": np.repeat(np.arange(23, dtype=np.int64), 5)[:100],
                                 "k2": np.tile(np.arange(-2, 3, dtype=np.int64), 23)[:100], "d1": rng2.randn(100)})
        w2 = orc.broadcast_merge_general(two, dim2, "left", 4, on=["key", "k2"])
        assert list(o["merge_two_keys"].columns) == list(w2.columns) and _same(o["merge_two_keys"].to_numpy(), w2.to_numpy())
        wf = vals[vals["c0"] > 0.0]
        assert list(o["filter"].index) == list(wf.index) and _same(o["filter"].to_numpy(), wf.to_numpy())
        wd = vals.dropna()
        assert list(o["dropna"].index) == list(wd.index) and _same(o["dropna"].to_numpy(), wd.to_numpy())
        assert int(np.asarray(o["nunique"]).ravel()[0]) == pdf["key"].nunique()
        assert np.isclose(o["sum_of_scaled_sums"], (vals.sum() * 2.0).sum(), rtol=1e-12, atol=0)
        assert np.isclose(o["max_of_means"], vals.mean().max(), rtol=1e-12, atol=0)
        assert o["count_positive_sums"] == int((vals.sum() > 0).sum())
        assert o["dd_last"].equals(pdf.drop_duplicates(subset=["key"], keep="last"))
        assert o["dd_series"].equals(pdf["key"].drop_duplicates())
        assert np.allclose(o["dd_then_sum"].to_numpy(), pdf.drop_duplicates(subset=["key"])[["c0", "c1"]].sum().to_numpy(), rtol=0, atol=1e-9)
        wsrt = vals.sort_values("c1", kind="stable")
        assert list(o["sort"].index) == list(wsrt.index) and _same(o["sort"].to_numpy(), wsrt.to_numpy())
    # the group table is split by key range: both ranks own a part, together all 23 groups
    assert sum(o["gb_local_sum"] for o in outs) == pdf["key"].nunique() and all(o["gb_local_sum"] > 0 for o in outs)
    assert all(o["gb_job_sum"] == pdf["key"].nunique() for o in outs)


def test_results_are_released_without_the_cycle_collector(modin_b200_execution, cpu_device):
    """A result frame must give its device buffers back when the last user reference goes -- not at the next run of
    Python's cycle collector.  The reference's frames reference themselves when their labels or dtypes are lazy
    (``ModinIndex(self, axis)``, df.py:526 / 542; ``DtypesDescriptor(parent_df=self)``, df.py:428-431); on the
    CPU engines that only delays the release of host memory, here it pinned 32 GB of HBM per ``df.cumsum()`` call
    (bench run of round 2: out of memory after five steps with the collector paused)."""
    import gc
    import weakref

    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: host-logic check for the CPU device double")
    _ns, mpd = modin_b200_execution
    pdf = synth.host_frame(3000, 4, seed=1, nan_per_64k=2000, key_modulus=10)
    df = mpd.DataFrame(pdf)
    vals = df[["c0", "c1", "c2", "c3"]]
    dim = mpd.DataFrame(pandas.DataFrame({"key": np.arange(10, dtype=np.int64), "w": np.arange(10) * 0.5}))
    gb = df.groupby("key")
    cases = {
        "x * s + t": lambda: vals * 2.0 + 1.0, "abs": lambda: vals.abs(), "cumsum": lambda: vals.cumsum(),
        "ffill": lambda: vals.ffill(), "groupby.sum": lambda: gb.sum(), "groupby.agg(dict)": lambda: gb.agg({"c0": "sum", "c1": "max"}),
        "merge": lambda: df.merge(dim, on="key", how="left"), "filter": lambda: vals[vals["c0"] > 0.0],
        "sort_values": lambda: vals.sort_values("c1"), "a + b": lambda: vals + vals, "dropna": lambda: vals.dropna(),
    }  # fmt: skip
    for call in cases.values():  # first use: caches (join tables, key statistics) may legitimately keep things alive
        call()._query_compiler.finalize()
    gc.collect()
    gc.disable()
    try:
        kept = []
        for name, call in cases.items():
            r = call()
            r._query_compiler.finalize()
            blk = r._query_compiler._modin_frame._partitions[0, 0].get()
            probe = weakref.ref(blk.cols[-1].data)  # the last column is always a fresh buffer of this result
            del r, blk
            if probe() is not None:
                kept.append(name)
        assert not kept, f"still allocated after the last reference went: {kept}"
    finally:
        gc.enable()


def _fold_and_keys_sweep_job(rank, ws):
    """Tiny and empty shards for what was written late in round 2 and crosses ranks: the Fold carries, float-key and
    ``level=`` groupby, dictionary aggregation -- through real ``modin.pandas`` on the numpy device double."""
    import sys

    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import warnings

    warnings.filterwarnings("ignore")
    import cpu_double
    from modin_b200 import config, modin_plugin

    out = []
    with cpu_double.installed():
        modin_plugin.activate()
        import modin.config as cfg
        import modin.pandas as mpd

        cfg.NPartitions.put(2)
        config.NPartitions.put(2)
        P = lambda x: x._to_pandas()  # noqa: E731
        for case, n in enumerate((1, 2, 5, 64, 2003)):  # 1, 2 and 5 rows over 3 ranks: some shards are empty
            rng = np.random.RandomState(40 + case)
            pdf = pandas.DataFrame({"a": rng.randn(n), "b": rng.randn(n), "i": rng.randint(-9, 9, n).astype(np.int64)})
            pdf.loc[rng.rand(n) < 0.3, "a"] = np.nan
            pdf.iloc[: max(1, n // 2), 1] = np.nan  # the first half of "b" has nothing valid: carries of "nothing yet"
            df = mpd.DataFrame(pdf)
            res = {"n": n}
            for name in ("cumsum", "cummax", "cummin", "ffill"):
                res[name] = P(getattr(df, name)())
            fvals = pdf[["a", "b"]]  # group sums / maxima aggregate float64 value columns
            fk = fvals.assign(fk=np.where(rng.rand(n) < 0.2, np.nan, np.round(rng.randn(n), 0) / 2.0))
            res["fk_frame"] = fk
            res["fk_sum"] = P(mpd.DataFrame(fk).groupby("fk").sum())
            lab = fvals.set_axis(pandas.Index(rng.randint(0, 4, n).astype(np.int64), name="lab"), axis=0)
            res["lab_frame"] = lab
            res["lab_max"] = P(mpd.DataFrame(lab).groupby(level=0).max())
            out.append((pdf, res))
    return out


def test_fold_and_key_kinds_sweep_across_three_ranks():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: tools/dist_check.py covers the plug-in under NCCL")
    from tests.test_dist_gloo import _run

    for rank_out in _run(_fold_and_keys_sweep_job, ws=3):
        for pdf, res in rank_out:
            n = res["n"]
            got, want = res["cumsum"], pdf.cumsum()
            assert list(got.index) == list(want.index) and np.allclose(got.to_numpy(), want.to_numpy(), rtol=0, atol=1e-9, equal_nan=True), n
            for name in ("cummax", "cummin", "ffill"):
                assert res[name].equals(getattr(pdf, name)()), (n, name)
            want = res["fk_frame"].groupby("fk").sum()
            assert np.array_equal(res["fk_sum"].index.to_numpy(), want.index.to_numpy()), n
            assert np.allclose(res["fk_sum"].to_numpy(), want.to_numpy(), rtol=0, atol=1e-9, equal_nan=True), n
            want = res["lab_frame"].groupby(level=0).max()
            assert np.array_equal(res["lab_max"].index.to_numpy(), want.index.to_numpy()) and res["lab_max"].index.name == "lab", n
            assert np.array_equal(res["lab_max"].to_numpy(), want.to_numpy(), equal_nan=True), n
