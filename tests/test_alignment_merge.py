"""Row-label alignment (the reindexing half of ``PandasDataframe._copartition``, df.py:3709-3848) and the general
broadcast merge (many-to-many keys, ``left_on`` / ``right_on``; storage_formats/pandas/merge.py:139-168), against golden
vectors produced by the unmodified reference (tests/golden/ext4_align_m2m.npz).

The same checks run three ways: through the mirror on the numpy device double (host logic, ``-m "not gpu"``), through
the mirror on a B200 and through the real ``modin.pandas`` with the plug-in on a B200 (``-m gpu``).  Everything here is
index / copy work, so the bar is bit-exact (NaN == NaN)."""

import os
import sys

import numpy as np
import pandas
import pytest

from modin_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
REF = os.path.join(ROOT, "oracle", "_ref")


def _same(got, want, what):
    g, w = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert g.shape == w.shape, f"{what}: shape {g.shape} vs {w.shape}"
    ok = (g.view(np.uint64) == w.view(np.uint64)) | (np.isnan(g) & np.isnan(w))
    assert ok.all(), f"{what}: {np.count_nonzero(~ok)} values differ"


def ext4_checks(pdm, real_modin=False):
    if GOLDEN not in sys.path:
        sys.path.insert(0, GOLDEN)
    from make_golden import fourth_batch_frames

    z = np.load(os.path.join(GOLDEN, "ext4_align_m2m.npz"), allow_pickle=False)
    A, B, Bp, fact, dim, dim_u = fourth_batch_frames(synth)
    a, b, bp_ = pdm.DataFrame(A), pdm.DataFrame(B), pdm.DataFrame(Bp)
    P = lambda x: x._to_pandas()  # noqa: E731
    r = P(a + b)
    assert np.array_equal(r.index.to_numpy(), z["add_index"])
    _same(r.to_numpy(), z["add"], "a + b on partly overlapping, permuted labels")
    r = P(a * b + a)
    assert np.array_equal(r.index.to_numpy(), z["mul_add_index"])
    _same(r.to_numpy(), z["mul_add"], "a * b + a")
    r = P(a < bp_)
    assert np.array_equal(r.index.to_numpy(), z["lt_index"])
    _same(r.to_numpy().astype(np.float64), z["lt"], "a < b' (same labels, permuted)")
    x = pdm.DataFrame(A)
    x["d"] = b["c0"]
    _same(P(x).to_numpy(), z["setitem"], "df['d'] = series on other labels")
    r = P(a[bp_["c0"] > 0])
    assert np.array_equal(r.index.to_numpy(), z["mask_index"])
    _same(r.to_numpy(), z["mask"], "df[mask on permuted labels]")
    r = P(pdm.concat([a, bp_.rename(columns={"c0": "x", "c1": "y", "c2": "z"})], axis=1))
    assert np.array_equal(r.index.to_numpy(), z["cat1_index"])
    _same(r.to_numpy(), z["cat1"], "concat(axis=1) on permuted labels")
    f, d, du = pdm.DataFrame(fact), pdm.DataFrame(dim), pdm.DataFrame(dim_u)
    for how in ("left", "inner"):
        r = P(f.merge(d, on="key", how=how))
        assert list(r.columns) == list(z[f"m2m_{how}_cols"])
        _same(r.to_numpy(dtype=np.float64), z[f"m2m_{how}"], f"many-to-many merge {how}")
        assert isinstance(r.index, pandas.RangeIndex) or np.array_equal(r.index.to_numpy(), np.arange(len(r)))
    r = P(f.merge(du, left_on="key", right_on="k", how="left"))
    assert list(r.columns) == list(z["lr_on_cols"])
    _same(r.to_numpy(dtype=np.float64), z["lr_on"], "merge left_on / right_on")
    # pandas' errors for labels that cannot be aligned
    if not real_modin:
        with pytest.raises(pandas.errors.IndexingError):
            a[b["c0"] > 0]  # the mask does not cover every row label of the frame
    pd_dup = pandas.DataFrame({"c0": [1.0, 2.0, 3.0]}, index=[0, 0, 1])
    pd_small = pandas.DataFrame({"c0": [1.0, 2.0, 3.0]}, index=[2, 1, 0])
    dup_labels, small = pdm.DataFrame(pd_dup), pdm.DataFrame(pd_small)
    if real_modin:  # Modin computes positional indexers on the host for repeated labels (df.py:2030-2072)
        r = P(small + dup_labels)
        w = pd_small + pd_dup
        assert list(r.index) == list(w.index)
        _same(r.to_numpy(), w.to_numpy(), "alignment with repeated labels")
    else:
        with pytest.raises(ValueError):
            P(small + dup_labels)  # the mirror refuses: "cannot reindex on an axis with duplicate labels"


def test_alignment_and_general_merge_on_the_double(cpu_device):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu-marked tests")
    import modin_b200.pandas as bpd
    from modin_b200 import config

    old = config.NPartitions.get()
    config.NPartitions.put(4)
    try:
        ext4_checks(bpd)
    finally:
        config.NPartitions.put(old)


@pytest.mark.gpu
def test_alignment_and_general_merge_on_b200():
    import modin_b200.pandas as bpd
    from modin_b200 import _lib, config

    lib = _lib.load()
    before = lib.mb200_launch_count()
    old = config.NPartitions.get()
    config.NPartitions.put(4)
    try:
        ext4_checks(bpd)
    finally:
        config.NPartitions.put(old)
    assert lib.mb200_launch_count() > before


def _modin(nparts=4):
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import warnings

    warnings.filterwarnings("ignore")
    from modin_b200 import config, modin_plugin

    modin_plugin.activate()
    import modin.config as cfg
    import modin.pandas as mpd

    cfg.NPartitions.put(nparts)
    config.NPartitions.put(nparts)
    return mpd


needs_modin = pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "modin")), reason="reference Modin not installed under oracle/_ref")


@needs_modin
def test_alignment_and_general_merge_under_real_modin_on_the_double(cpu_device):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu-marked test")
    ext4_checks(_modin(), real_modin=True)


@needs_modin
@pytest.mark.gpu
def test_alignment_and_general_merge_under_real_modin_on_b200():
    from modin_b200 import _lib

    lib = _lib.load()
    before = lib.mb200_launch_count()
    ext4_checks(_modin(), real_modin=True)
    assert lib.mb200_launch_count() > before


@pytest.mark.gpu
def test_many_to_many_expansion_at_scale():
    """2^22 fact rows against 3e5 dim rows with up to 4 copies of a key: row pairs equal numpy's (bit-exact)."""
    from modin_b200 import ops
    from modin_b200.block import DeviceColumn

    rng = np.random.RandomState(3)
    dk = rng.randint(0, 100_000, size=300_000).astype(np.int64)
    fk = rng.randint(0, 120_000, size=1 << 22).astype(np.int64)
    for keep in (True, False):
        lr, rr, misses = ops.expand_matches(DeviceColumn.from_numpy(fk), DeviceColumn.from_numpy(dk), keep_misses=keep)
        order = np.argsort(dk, kind="stable")
        ks = dk[order]
        lo, hi = np.searchsorted(ks, fk, "left"), np.searchsorted(ks, fk, "right")
        cnt = hi - lo
        assert misses == int((cnt == 0).sum())
        out_cnt = np.where(cnt > 0, cnt, 1 if keep else 0)
        left = np.repeat(np.arange(len(fk)), out_cnt)
        offs = np.cumsum(out_cnt) - out_cnt
        src = np.repeat(lo, out_cnt) + (np.arange(len(left)) - np.repeat(offs, out_cnt))
        right = np.where(np.repeat(cnt > 0, out_cnt), order[np.minimum(src, len(order) - 1)], -1)
        assert np.array_equal(lr.to_numpy(), left) and np.array_equal(rr.to_numpy(), right)


# ---- range-partitioning shuffle (pm.shuffle_partitions, partition_manager.py:1937-2052) --------------------------
def _shuffle_checks(bpd, n):
    from modin_b200 import config
    from modin_b200.shuffle import DevShuffleFunctions, DevSortBlock

    old = config.NPartitions.get()
    config.NPartitions.put(4)
    try:
        pdf = synth.host_frame(n, 3, seed=5, nan_per_64k=3000, key_modulus=777)
        df = bpd.DataFrame(pdf)
        frame = df._query_compiler._modin_frame
        pm = frame._partition_mgr_cls
        # the classmethod itself: 4 key ranges, disjoint and in key order, every row exactly once
        sf = DevShuffleFunctions(1, ascending=True, ideal_num_new_partitions=4)  # column 1 = c0
        parts = pm.shuffle_partitions(frame._partitions, 0, sf, DevSortBlock(1, True))
        assert parts.shape == (4, 1) and len(sf.pivots) == 3
        blocks = [p[0].get() for p in parts]
        assert sum(b.nrows for b in blocks) == n
        pieces = [b.to_pandas() for b in blocks]
        keys = [p["c0"].to_numpy() for p in pieces]
        tops = [np.nanmax(k) for k in keys if len(k) and not np.isnan(k).all()]
        lows = [np.nanmin(k) for k in keys if len(k) and not np.isnan(k).all()]
        assert all(t <= l for t, l in zip(tops[:-1], lows[1:])), "key ranges overlap"
        got = pandas.concat(pieces)
        want = pdf.sort_values("c0", kind="stable")
        assert got.index.equals(want.index), "rows out of stable key order"
        assert np.array_equal(got.to_numpy().view(np.uint64), want.to_numpy().view(np.uint64))
        # through the API, both directions, float and int keys, labels kept or renumbered
        for by, asc in (("c1", False), ("key", True), ("key", False)):
            got = df.sort_values(by, ascending=asc)._to_pandas()
            want = pdf.sort_values(by, ascending=asc, kind="stable")
            assert got.index.equals(want.index) and np.array_equal(got.to_numpy().view(np.uint64), want.to_numpy().view(np.uint64)), (by, asc)
        got = df.sort_values("c0", ignore_index=True)._to_pandas()
        want = pdf.sort_values("c0", ignore_index=True, kind="stable")
        assert got.index.equals(want.index) and np.array_equal(got.to_numpy().view(np.uint64), want.to_numpy().view(np.uint64))
    finally:
        config.NPartitions.put(old)


def test_shuffle_partitions_on_the_double(cpu_device):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu-marked test")
    import modin_b200.pandas as bpd

    _shuffle_checks(bpd, 300_000)


@pytest.mark.gpu
def test_shuffle_partitions_on_b200():
    import modin_b200.pandas as bpd

    _shuffle_checks(bpd, 1 << 21)


# ---- groupby(as_index=False) (alg/groupby.py:278-294) and read_parquet -> Arrow -> device ---------------------------
def _as_index_and_parquet_checks(pdm, tmp_path, real_modin):
    pdf = synth.host_frame(5000, 3, seed=2, nan_per_64k=2000, key_modulus=37)
    for agg in ("sum", "count", "max"):
        got = getattr(pdm.DataFrame(pdf).groupby("key", as_index=False), agg)()._to_pandas()
        want = getattr(pdf.groupby("key", as_index=False), agg)()
        assert list(got.columns) == list(want.columns) and got.index.equals(want.index), agg
        assert np.allclose(got.to_numpy(dtype=np.float64), want.to_numpy(dtype=np.float64), rtol=0, atol=1e-9, equal_nan=True), agg
    # several int64 keys (packed into one order-preserving int64 on the device, groupkeys.py)
    pdf["k2"] = synth.gen_i64(5000, 99, 1, 5) * 10 - 20
    for agg in ("sum", "count", "min"):
        got = getattr(pdm.DataFrame(pdf).groupby(["key", "k2"]), agg)()._to_pandas()
        want = getattr(pdf.groupby(["key", "k2"]), agg)()
        assert got.index.equals(want.index) and list(got.columns) == list(want.columns), agg
        assert np.allclose(got.to_numpy(dtype=np.float64), want.to_numpy(dtype=np.float64), rtol=0, atol=1e-9, equal_nan=True), agg
    if real_modin:
        got = pdm.DataFrame(pdf).groupby(["key", "k2"], as_index=False).sum()._to_pandas()
        want = pdf.groupby(["key", "k2"], as_index=False).sum()
        assert list(got.columns) == list(want.columns) and np.allclose(got.to_numpy(dtype=np.float64), want.to_numpy(dtype=np.float64), rtol=0, atol=1e-9)
    # dictionary aggregations (qc._groupby_dict_reduce, qc.py:3876-3970): one device aggregation per distinct function
    spec = {"c2": "mean", "c0": "sum", "c1": "max"}
    for by, kw in (("key", {}), ("key", {"as_index": False}), (["key", "k2"], {})):
        if not real_modin and kw:
            continue
        got = pdm.DataFrame(pdf).groupby(by, **kw).agg(spec)._to_pandas()
        want = pdf.groupby(by, **kw).agg(spec)
        assert list(got.columns) == list(want.columns) and got.index.equals(want.index), (by, kw)
        assert np.allclose(got.to_numpy(dtype=np.float64), want.to_numpy(dtype=np.float64), rtol=0, atol=1e-9, equal_nan=True), (by, kw)
    fl = pdf[["key", "c0", "c1"]]  # min / max / sum aggregate float64 value columns
    assert pdm.DataFrame(fl).groupby("key").agg("min")._to_pandas().equals(fl.groupby("key").agg("min"))
    with pytest.raises(NotImplementedError):
        pdm.DataFrame(pdf).groupby("key").agg({"c0": "median"})
    if real_modin:
        path = os.path.join(str(tmp_path), "frame.parquet")
        pdf.to_parquet(path)
        got = pdm.read_parquet(path, columns=["key", "c1"])
        from modin_b200.block import DeviceBlock

        assert all(isinstance(p.get(), DeviceBlock) for p in got._query_compiler._modin_frame._partitions.flatten())
        assert got._to_pandas().equals(pdf[["key", "c1"]])
        with pytest.raises(NotImplementedError):
            pdm.read_parquet(path, filters=[("key", ">", 3)])


def test_as_index_false_on_the_double(cpu_device, tmp_path):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu-marked test")
    import modin_b200.pandas as bpd

    _as_index_and_parquet_checks(bpd, tmp_path, False)


@needs_modin
def test_as_index_false_and_read_parquet_under_real_modin_on_the_double(cpu_device, tmp_path):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu-marked test")
    _as_index_and_parquet_checks(_modin(), tmp_path, True)


@needs_modin
@pytest.mark.gpu
def test_as_index_false_and_read_parquet_under_real_modin_on_b200(tmp_path):
    import modin_b200.pandas as bpd

    _as_index_and_parquet_checks(bpd, tmp_path, False)
    _as_index_and_parquet_checks(_modin(), tmp_path, True)
