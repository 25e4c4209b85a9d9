"""GPU parity of boolean row selection / dropna (``df[mask]``): mask -> ranked compaction -> one gather per column.

Written after this round's GPU budget was spent, so it has only run on the CPU device double so far
(tests/test_host_stack_cpu.py::test_boolean_row_selection_and_dropna).  Every kernel it reaches is covered by
other GPU tests (bool widening and logical ops: test_boolean_pipelines_on_device; compaction and gather: the
inner-merge tests); the file sorts last so that a surprise here cannot hide the rest of the suite behind ``-x``.

The same holds for the later additions in this file (isin, concat, astype / DataFrame.nunique, drop_duplicates, the
ext2 and ext3 golden vectors): NOT yet run on a B200, only on the double.  concat launches nothing itself; astype
reuses the true-division and widening-copy kernels that the var / std and bool-sum GPU tests already reach;
drop_duplicates is sort + elementwise compare + compaction + gather, each reached by sort_values / row selection
tests -- the one new thing it does to a kernel is hand the elementwise compare two views shifted by one row (8-byte
aligned, not 32), which elementwise.cu routes to its scalar sweep (``aligned32`` test on every operand).
"""

import numpy as np
import pytest

from modin_b200 import synth

pytestmark = pytest.mark.gpu


def _exact(got, want, what):
    g, w = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert g.shape == w.shape, f"{what}: shape {g.shape} vs {w.shape}"
    assert ((g.view(np.uint64) == w.view(np.uint64)) | (np.isnan(g) & np.isnan(w))).all(), what


def test_boolean_row_selection_and_dropna_on_device():
    import modin_b200.pandas as bpd
    from modin_b200 import config

    old = config.NPartitions.get()
    config.NPartitions.put(4)
    try:
        pdf = synth.host_frame(100_003, 3, seed=21, nan_per_64k=6000, key_modulus=9)
        df = bpd.DataFrame(pdf)
        for got, want in (
            (df[df["c0"] > 0.5], pdf[pdf["c0"] > 0.5]),
            (df[(df["c0"] > 0.0) & (df["c1"] < 0.0)], pdf[(pdf["c0"] > 0.0) & (pdf["c1"] < 0.0)]),
            (df[df["key"] == 3], pdf[pdf["key"] == 3]),
            (df[df["c2"] > 100.0], pdf[pdf["c2"] > 100.0]),
            (df.dropna(), pdf.dropna()),
            (df.dropna(how="all", subset=["c0", "c1"]), pdf.dropna(how="all", subset=["c0", "c1"])),
        ):
            g = got._to_pandas()
            assert np.array_equal(g.index.to_numpy(), want.index.to_numpy()) and list(g.columns) == list(want.columns)
            _exact(g.to_numpy(dtype=np.float64), want.to_numpy(dtype=np.float64), "row selection")
        sel = df[df["c0"] > 0.0]
        want = pdf[pdf["c0"] > 0.0]
        assert np.allclose(sel.sum().to_numpy(), want.sum().to_numpy(), rtol=0, atol=1e-8)
        _exact(sel.groupby("key").count()._to_pandas().to_numpy(), want.groupby("key").count().to_numpy(), "count after filter")
    finally:
        config.NPartitions.put(old)


def test_pipeline_filter_derive_aggregate_on_device():
    """setitem / assign / drop / rename / head / tail are metadata over shared buffers; a whole pipeline stays on
    the device: filter -> derived column -> groupby."""
    import modin_b200.pandas as bpd
    from modin_b200 import config

    old = config.NPartitions.get()
    config.NPartitions.put(4)
    try:
        pdf = synth.host_frame(50_003, 3, seed=31, nan_per_64k=1000, key_modulus=5)
        df = bpd.DataFrame(pdf)
        out = df[df["c0"] > 0.0].assign(g=lambda x: x["c1"] * x["c2"]).groupby("key").sum()._to_pandas()
        w = pdf[pdf["c0"] > 0.0].assign(g=lambda x: x["c1"] * x["c2"]).groupby("key").sum()
        assert list(out.columns) == list(w.columns) and np.allclose(out.to_numpy(), w.to_numpy(), rtol=0, atol=1e-8)
        d2 = df.copy()
        d2["c1"] = d2["c0"] + d2["c2"]
        want = pdf.copy()
        want["c1"] = want["c0"] + want["c2"]
        _exact(d2._to_pandas().to_numpy(dtype=np.float64), want.to_numpy(dtype=np.float64), "setitem replace")
        for n in (0, 7, 12_501, 50_003):
            _exact(df.head(n)._to_pandas().to_numpy(dtype=np.float64), pdf.head(n).to_numpy(dtype=np.float64), f"head {n}")
            _exact(df.tail(n)._to_pandas().to_numpy(dtype=np.float64), pdf.tail(n).to_numpy(dtype=np.float64), f"tail {n}")
    finally:
        config.NPartitions.put(old)


def test_isin_is_a_join_probe_on_device():
    import modin_b200.pandas as bpd

    pdf = synth.host_frame(30_011, 2, seed=5, key_modulus=500)
    df = bpd.DataFrame(pdf)
    vals = [3, 7, 7, 41, -2, 100_000]
    got = df[["key"]].isin(vals)._to_pandas()
    assert np.array_equal(got.to_numpy(), pdf[["key"]].isin(vals).to_numpy())
    sel = df[df["key"].isin([1, 2, 3])]._to_pandas()
    w = pdf[pdf["key"].isin([1, 2, 3])]
    assert np.array_equal(sel.index.to_numpy(), w.index.to_numpy())
    _exact(sel.to_numpy(dtype=np.float64), w.to_numpy(dtype=np.float64), "filter by isin")


def test_baseline_config0_abs_and_sum_at_its_own_size():
    """BASELINE.json configs[0] -- ``df.abs()`` + ``df.sum()`` on 1e6 x 4 float64, the reference's own CPU-runnable
    case -- at exactly that size against the oracle (NPartitions=4): abs bit-exact, the sum within the fp64 tolerance
    the north star states, 4 * log2(n) * 2**-53 * sum|x| (same code path as test_against_oracle_various_shapes, which
    stops at 262144 rows)."""
    import math

    import modin_b200.pandas as bpd
    from modin_b200 import config
    from oracle import reference_path as orc

    old = config.NPartitions.get()
    config.NPartitions.put(4)
    try:
        n, W = 1_000_000, 4
        pdf = synth.host_frame(n, W, seed=5, nan_per_64k=500)
        df = bpd.DataFrame(pdf)
        _exact(df.abs()._to_pandas().to_numpy(), orc.df_abs(pdf, 4).to_numpy(), "abs 1e6 x 4")
        got, want = np.asarray(df.sum(), dtype=np.float64), orc.df_sum(pdf, 4).to_numpy()
        tol = 4.0 * math.log2(n) * 2.0**-53 * np.nansum(np.abs(pdf.to_numpy()), axis=0)
        assert got.shape == want.shape == (W,) and (np.abs(got - want) <= tol).all(), (got - want, tol)
        gabs = np.asarray(df.abs().sum(), dtype=np.float64)  # the config's two operations chained
        assert (np.abs(gabs - orc.df_sum(orc.df_abs(pdf, 4), 4).to_numpy()) <= tol).all()
    finally:
        config.NPartitions.put(old)


def test_concat_on_device():
    """concat(axis=0) lines up row partitions (labels restart per input unless ignore_index); axis=1 is hstack.
    No kernel of its own: what is checked on the device is that operators run over the lined-up partitions."""
    import pandas

    import modin_b200.pandas as bpd
    from modin_b200 import config

    old = config.NPartitions.get()
    config.NPartitions.put(4)
    try:
        pa = synth.host_frame(40_003, 3, seed=41, nan_per_64k=1000, key_modulus=5)
        pb = synth.host_frame(20_017, 3, seed=42, nan_per_64k=1000, key_modulus=5)
        a, b = bpd.DataFrame(pa), bpd.DataFrame(pb)
        for ignore in (False, True):
            got = bpd.concat([a, b, a], ignore_index=ignore)._to_pandas()
            want = pandas.concat([pa, pb, pa], ignore_index=ignore)
            assert np.array_equal(got.index.to_numpy(), want.index.to_numpy()) and list(got.columns) == list(want.columns)
            _exact(got.to_numpy(dtype=np.float64), want.to_numpy(dtype=np.float64), "concat rows")
        cat, wcat = bpd.concat([a, b], ignore_index=True), pandas.concat([pa, pb], ignore_index=True)
        _exact((cat * 2.0)._to_pandas().to_numpy(dtype=np.float64), (wcat * 2.0).to_numpy(dtype=np.float64), "map over concat")
        g, wg = cat.groupby("key").sum()._to_pandas(), wcat.groupby("key").sum()
        assert np.array_equal(g.index.to_numpy(), wg.index.to_numpy()) and np.allclose(g.to_numpy(), wg.to_numpy(), rtol=0, atol=1e-8)
        right = a[["c0", "c1"]].rename(columns={"c0": "x", "c1": "y"})
        wide = bpd.concat([a, right], axis=1)._to_pandas()
        wwide = pandas.concat([pa, pa[["c0", "c1"]].rename(columns={"c0": "x", "c1": "y"})], axis=1)
        assert list(wide.columns) == list(wwide.columns)
        _exact(wide.to_numpy(dtype=np.float64), wwide.to_numpy(dtype=np.float64), "concat columns")
    finally:
        config.NPartitions.put(old)


def test_astype_and_frame_nunique_on_device():
    """int64 / bool -> float64 through the true-division kernel (round to nearest even above 2**53, as numpy),
    bool -> int64 through the widening copy; DataFrame.nunique = rows of one group table per int64 column."""
    import pandas

    import modin_b200.pandas as bpd

    rng = np.random.default_rng(51)
    n = 60_007
    pdf = pandas.DataFrame({
        "k": rng.integers(-7, 7, n),
        "big": rng.integers(-(2**62), 2**62, n),
        "x": rng.standard_normal(n),
        "flag": rng.integers(0, 2, n).astype(bool),
    })  # fmt: skip
    pdf.loc[::97, "x"] = np.nan
    df = bpd.DataFrame(pdf)
    got, want = df.astype("float64"), pdf.astype("float64")
    assert list(got.dtypes) == list(want.dtypes)
    _exact(got._to_pandas().to_numpy(), want.to_numpy(), "astype float64")
    got = df.astype({"k": np.float64, "flag": "int64"})._to_pandas()
    want = pdf.astype({"k": np.float64, "flag": "int64"})
    for c in want.columns:
        assert got[c].dtype == want[c].dtype, c
        _exact(got[c].to_numpy(dtype=np.float64), want[c].to_numpy(dtype=np.float64), f"astype dict {c}")
    assert np.array_equal(got["big"].to_numpy(), want["big"].to_numpy())  # untouched int64 column, exact
    with pytest.raises(NotImplementedError):
        df.astype("int64")
    nu, wnu = df[["k", "big"]].nunique(), pdf[["k", "big"]].nunique()
    assert list(nu.index) == list(wnu.index) and list(nu) == list(wnu)


def test_second_batch_vs_reference_golden(golden_dir):
    """The same operations against golden vectors produced by the UNMODIFIED reference (tests/golden/ext2_*.npz):
    logical ops, any / all, bool sums, isin, boolean row selection, dropna, multi-column groupby, dict aggregation,
    value_counts, nunique."""
    import glob
    import os

    import modin_b200.pandas as bpd
    from modin_b200 import config

    old = config.NPartitions.get()
    config.NPartitions.put(4)
    try:
        files = sorted(glob.glob(os.path.join(golden_dir, "ext2_*.npz")))
        assert files
        for f in files:
            z = np.load(f, allow_pickle=False)
            n, seed, nan, G = (int(x) for x in z["meta"])
            pdf = synth.host_frame(n, 3, seed=seed, nan_per_64k=nan, key_modulus=G)
            pdf["k2"] = synth.gen_i64(n, 99, 1, 5) * 10 - 20
            df = bpd.DataFrame(pdf)
            v = df[["c0", "c1", "c2"]]
            band = (v > 0.0) & (v < 1.0)
            assert np.array_equal(band._to_pandas().to_numpy(), z["band"])
            assert np.array_equal(((v > 0.5) | (v < -0.5))._to_pandas().to_numpy(), z["bor"])
            assert np.array_equal(((v > 0.0) ^ (v > 1.0))._to_pandas().to_numpy(), z["bxor"])
            assert np.array_equal((~band)._to_pandas().to_numpy(), z["bnot"])
            assert np.array_equal(band.any().to_numpy(), z["any"]) and np.array_equal((v > -100.0).all().to_numpy(), z["all_true"])
            assert np.array_equal(band.sum().to_numpy(), z["boolsum"])
            assert np.allclose(band.mean().to_numpy(), z["boolmean"], rtol=1e-12, atol=0)
            assert np.array_equal(df[["key", "k2"]].isin([3, 7, -20, 30])._to_pandas().to_numpy(), z["isin"])
            sel = df[df["c0"] > 0.5]._to_pandas()
            assert np.array_equal(sel.index.to_numpy(), z["sel_index"])
            _exact(sel.to_numpy(dtype=np.float64), z["sel"], "filter")
            dn = df.dropna()._to_pandas()
            assert np.array_equal(dn.index.to_numpy(), z["dropna_index"])
            _exact(dn.to_numpy(dtype=np.float64), z["dropna"], "dropna")
            mk = df.groupby(["key", "k2"]).sum()._to_pandas()
            assert np.array_equal(mk.index.get_level_values(0).to_numpy(), z["mk_k1"])
            assert np.array_equal(mk.index.get_level_values(1).to_numpy(), z["mk_k2"])
            assert np.allclose(mk.to_numpy(), z["mk_sum"], rtol=0, atol=1e-9)
            da = df.groupby("key").agg({"c1": "max", "c0": "sum", "c2": "count"})._to_pandas()
            assert np.array_equal(da.index.to_numpy(), z["dict_keys"])
            assert np.allclose(da.to_numpy(dtype=np.float64), z["dict_agg"], rtol=0, atol=1e-9)
            vc = df["key"].value_counts()._to_pandas()
            assert np.array_equal(vc.to_numpy(), z["vc_counts"])
            assert dict(zip(vc.index, vc.to_numpy())) == dict(zip(z["vc_keys"], z["vc_counts"]))
            assert df["key"].nunique() == int(z["nunique"][0])
    finally:
        config.NPartitions.put(old)


def test_third_batch_vs_reference_golden(golden_dir):
    """drop_duplicates, concat, astype, DataFrame.nunique against golden vectors produced by the UNMODIFIED reference
    (tests/golden/ext3_*.npz); inputs come from the generator's own helper (no reference needed to build them)."""
    import glob
    import importlib.util
    import os

    import modin_b200.pandas as bpd
    from modin_b200 import config

    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(golden_dir, "make_golden.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    old = config.NPartitions.get()
    config.NPartitions.put(4)
    try:
        files = sorted(glob.glob(os.path.join(golden_dir, "ext3_*.npz")))
        assert files
        num = ["key", "k2", "c0", "c1", "c2"]
        for f in files:
            z = np.load(f, allow_pickle=False)
            n, nb, nan, G = (int(x) for x in z["meta"])
            pdf, pb = gen.third_batch_frames(synth, n, nb, nan, G)
            df, db = bpd.DataFrame(pdf), bpd.DataFrame(pb)
            for keep in ("first", "last"):
                r = df[num].drop_duplicates(subset=["key"], keep=keep)._to_pandas()
                assert np.array_equal(r.index.to_numpy(), z[f"dd_{keep}_index"]), keep
                _exact(r.to_numpy(dtype=np.float64), z[f"dd_{keep}"], f"drop_duplicates {keep}")
            r = df[num].drop_duplicates(subset=["k2"], keep="last", ignore_index=True)._to_pandas()
            assert np.array_equal(r.index.to_numpy(), z["dd_k2_ignore_index"])
            _exact(r.to_numpy(dtype=np.float64), z["dd_k2_ignore"], "drop_duplicates ignore_index")
            r = df["k2"].drop_duplicates()._to_pandas()
            assert np.array_equal(r.index.to_numpy(), z["dd_series_index"])
            assert np.array_equal(np.asarray(r).ravel(), z["dd_series"])
            for ig in (False, True):
                r = bpd.concat([df[num], db[num], df[num]], ignore_index=ig)._to_pandas()
                assert np.array_equal(r.index.to_numpy(), z[f"cat0_ig{int(ig)}_index"]), ig
                _exact(r.to_numpy(dtype=np.float64), z[f"cat0_ig{int(ig)}"], f"concat rows ig={ig}")
            r = bpd.concat([df[num], df[["c0", "c1"]].rename(columns={"c0": "x", "c1": "y"})], axis=1)._to_pandas()
            assert list(r.columns) == list(z["cat1_cols"])
            _exact(r.to_numpy(dtype=np.float64), z["cat1"], "concat columns")
            r = df.astype("float64")
            assert all(t == np.float64 for t in r.dtypes)
            _exact(r._to_pandas().to_numpy(), z["astype_f64"], "astype float64")
            r = df.astype({"key": np.float64, "flag": "int64"})
            assert [str(t) for t in r.dtypes] == list(z["astype_dict_dtypes"])
            _exact(r._to_pandas().to_numpy(dtype=np.float64), z["astype_dict"], "astype mapping")
            _exact(df[["key", "k2", "big"]].astype("float64")._to_pandas().to_numpy(), z["astype_big"], "astype of large ints")
            r = df[["key", "k2", "big"]].nunique()
            assert list(r.index) == list(z["nunique_cols"]) and np.array_equal(np.asarray(r), z["nunique"])
    finally:
        config.NPartitions.put(old)


def test_late_additions_under_real_modin_on_b200():
    """The same astype / drop_duplicates / unique / concat / nunique / reset_index scenarios as
    tests/test_modin_plugin.py::test_late_additions_under_real_modin_cpu_double, through real ``modin.pandas`` with
    the B200 execution plugged in.  Needs the reference Modin under oracle/_ref (it travels with the snapshot)."""
    import importlib.util
    import os
    import sys
    import warnings

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ref = os.path.join(root, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref, "modin")):
        pytest.skip("reference Modin not installed under oracle/_ref")
    if ref not in sys.path:
        sys.path.insert(0, ref)
    warnings.filterwarnings("ignore")
    from modin_b200 import _lib, config, modin_plugin

    ns = modin_plugin.register()
    import modin
    import modin.config as cfg
    import modin.pandas as mpd

    modin.set_execution(engine="B200", storage_format="Arrow")
    cfg.NPartitions.put(4)
    spec = importlib.util.spec_from_file_location("plugin_scenarios", os.path.join(root, "tests", "test_modin_plugin.py"))
    scen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(scen)
    old = config.NPartitions.get()
    config.NPartitions.put(4)
    try:
        lib = _lib.load()
        before = lib.mb200_launch_count()
        scen._late_scenarios(mpd, ns)
        assert lib.mb200_launch_count() > before
    finally:
        config.NPartitions.put(old)
