"""Multi-GPU parity check, run under torchrun (one rank per GPU, NCCL):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29611 \
        tools/dist_check.py

Every rank builds the SAME seeded host frame, ingests only its row shard (pm.from_pandas shards by
rank), runs the hot-path templates through the public API and compares the gathered results with
the CPU oracle.  Exit code 0 = all checks passed on every rank.

``--api mirror`` (default: both) drives ``modin_b200.pandas``; ``--api modin`` drives the REAL ``modin.pandas``
(oracle/_ref) with the plug-in activated on every rank -- the same checks, plus the operations the plug-in refuses
on all ranks together.
"""
import math
import os
import sys

import numpy as np
import pandas

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from modin_b200 import config, dist, synth  # noqa: E402
from oracle import reference_path as orc  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

EPS = 2.0**-53


def exact(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and bool(((a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))).all())


def close(a, b, abs_sum, n):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    tol = 4 * max(1.0, math.log2(n)) * EPS * np.asarray(abs_sum, dtype=np.float64) + 1e-300
    return a.shape == b.shape and bool(((np.abs(a - b) <= tol) | (a == b) | (np.isnan(a) & np.isnan(b))).all())


def front_door(which):
    if which == "mirror":
        import modin_b200.pandas as bpd

        return bpd
    ref = os.path.join(ROOT, "oracle", "_ref")
    if ref not in sys.path:
        sys.path.insert(0, ref)
    import warnings

    warnings.filterwarnings("ignore")
    from modin_b200 import modin_plugin

    modin_plugin.activate()
    import modin.config as cfg
    import modin.pandas as mpd

    cfg.NPartitions.put(2)
    return mpd


def run_checks(bpd, tag, rank, fails):
    def P(x):
        return x._to_pandas() if hasattr(x, "_to_pandas") else x

    def check(name, ok):
        name = f"[{tag}] {name}"
        if not ok:
            fails.append(name)
        if rank == 0:
            print(("PASS " if ok else "FAIL ") + name, flush=True)

    n, W, G = 200_003, 5, 4_001
    pdf = synth.host_frame(n, W, seed=42, nan_per_64k=700, key_modulus=G)
    vals = pdf.drop(columns="key")
    df = bpd.DataFrame(pdf)  # this rank's shard only
    lo, hi = dist.shard_bounds(n)
    check("local shard length", len(df._query_compiler._modin_frame) == hi - lo)
    check("len(df) is the job-wide row count" if tag == "modin" else "len(df) is this rank's shard",
          len(df) == (n if tag == "modin" else hi - lo))
    dv = df[[f"c{i}" for i in range(W)]]
    NP = 4

    check("map abs (gathered, bit-exact)", exact(P(dv.abs()).to_numpy(), orc.df_abs(vals, NP).to_numpy()))
    check("fused a*b+c (gathered, bit-exact)",
          exact(P(dv * 1.25 + 0.5).to_numpy(), orc.a_mul_b_add_c(vals, 1.25, 0.5, NP).to_numpy()))
    abs_sum = np.nansum(np.abs(vals.to_numpy()), axis=0)
    check("tree_reduce sum (all_reduce)", close(np.asarray(P(dv.sum())), orc.df_sum(vals, NP).to_numpy(), abs_sum, n))
    check("tree_reduce count", exact(np.asarray(P(dv.count())), orc.df_count(vals, NP).to_numpy()))
    check("tree_reduce min", exact(np.asarray(P(dv.min())), orc.df_min(vals, NP).to_numpy()))
    check("tree_reduce max", exact(np.asarray(P(dv.max())), orc.df_max(vals, NP).to_numpy()))
    cnt = np.maximum(orc.df_count(vals, NP).to_numpy(), 1)
    check("tree_reduce mean", close(np.asarray(P(dv.mean())), orc.df_mean(vals, NP).to_numpy(), abs_sum / cnt, n))

    from modin_b200 import config as _cfg

    for dense, kind in ((True, "dense table + reduce-scatter"), (False, "hash tables + range exchange")):
        _cfg.GroupbyDenseKeys.put(dense)
        g = df.groupby("key")
        want = orc.groupby_reduce(pdf, "key", "sum", NP)
        got_local = g.sum()
        check(f"[{kind}] groupby: every rank owns a non-empty key range", len(got_local) > 0)
        got = P(got_local)  # gathers the per-rank key ranges in rank order
        gabs = vals.abs().groupby(pdf["key"]).sum().to_numpy()
        check(f"[{kind}] groupby keys globally sorted & complete", np.array_equal(got.index.to_numpy(), want.index.to_numpy()))
        check(f"[{kind}] groupby sum", close(got.to_numpy(), want.to_numpy(), gabs, n))
        check(f"[{kind}] groupby count", exact(P(g.count()).to_numpy(), orc.groupby_reduce(pdf, "key", "count", NP).to_numpy()))
        check(f"[{kind}] groupby size", exact(np.asarray(P(g.size())).ravel(), orc.groupby_reduce(pdf, "key", "size", NP).to_numpy().ravel()))
        gc = np.maximum(orc.groupby_reduce(pdf, "key", "count", NP).to_numpy(), 1)
        check(f"[{kind}] groupby mean", close(P(g.mean()).to_numpy(), orc.groupby_reduce(pdf, "key", "mean", NP).to_numpy(),
                                    gabs / gc, n))
        for agg in ("min", "max"):
            check(f"[{kind}] groupby {agg}", exact(P(getattr(g, agg)()).to_numpy(),
                                                 orc.groupby_reduce(pdf, "key", agg, NP).to_numpy()))
    _cfg.GroupbyDenseKeys.put(True)

    rng = np.random.RandomState(5)
    dim_keys = rng.permutation(G).astype(np.int64)[: int(G * 0.9)]
    dim = pandas.DataFrame({"key": dim_keys, "d0": synth.gen_f64(len(dim_keys), 11, 0)})
    mdim = bpd.DataFrame(dim)  # sharded too; combine() all-gathers it
    left = P(df.merge(mdim, on="key", how="left"))
    wl = orc.broadcast_merge(pdf, dim, "key", "left", NP)
    check("merge left (dim all_gathered)", list(left.columns) == list(wl.columns) and
          exact(left.to_numpy(dtype=np.float64), wl.to_numpy(dtype=np.float64)))
    inner = P(df.merge(mdim, on="key", how="inner"))
    wi = orc.broadcast_merge(pdf, dim, "key", "inner", NP)
    check("merge inner", exact(inner.to_numpy(dtype=np.float64), wi.to_numpy(dtype=np.float64)))

    # many-to-many merge (repeated dim keys) and the range-partitioning shuffle (sort_values) across ranks
    dup = pandas.DataFrame({"key": np.concatenate([dim_keys[:300], dim_keys[:120]]), "d1": np.arange(420, dtype=np.int64)})
    m2m = P(df.merge(bpd.DataFrame(dup), on="key", how="inner"))
    wm = orc.broadcast_merge_general(pdf, dup, "inner", NP, on="key")
    check("merge inner, repeated dim keys (many-to-many)", exact(m2m.to_numpy(dtype=np.float64), wm.to_numpy(dtype=np.float64)))
    two = pdf.assign(k2=(np.arange(n, dtype=np.int64) * 7) % 5 - 2)
    dim2 = pandas.DataFrame({"key": np.repeat(np.arange(G, dtype=np.int64), 5)[: 4 * G],
                             "k2": np.tile(np.arange(-2, 3, dtype=np.int64), G)[: 4 * G], "d1": rng.randn(4 * G)})
    mk, wmk = P(bpd.DataFrame(two).merge(bpd.DataFrame(dim2), on=["key", "k2"], how="left")), two.merge(dim2, on=["key", "k2"], how="left")
    check("merge on two key columns (packed keys)", list(mk.columns) == list(wmk.columns) and
          exact(mk.to_numpy(dtype=np.float64), wmk.to_numpy(dtype=np.float64)))
    srt = P(dv.sort_values("c1"))
    ws_ = vals.sort_values("c1", kind="stable")
    check("sort_values (range shuffle, all_to_all of rows)", list(srt.index) == list(ws_.index) and exact(srt.to_numpy(), ws_.to_numpy()))
    # drop_duplicates: the keys of each rank's own survivors are all-gathered, the result stays row-sharded
    for keep in ("first", "last"):
        dd, wdd = P(df.drop_duplicates(subset=["key"], keep=keep)), pdf.drop_duplicates(subset=["key"], keep=keep)
        check(f"drop_duplicates keep={keep} (survivor keys all_gathered)",
              list(dd.index) == list(wdd.index) and exact(dd.to_numpy(dtype=np.float64), wdd.to_numpy(dtype=np.float64)))
    if tag == "modin":  # the templates added late in round 2 are reached through Modin's own API
        # Fold: every rank scans its shard, the W column totals are all-gathered, carries are combined on the device
        cs, wcs = P(dv.cumsum()).to_numpy(), vals.cumsum().to_numpy()
        run_abs = np.cumsum(np.abs(np.nan_to_num(vals.to_numpy())), axis=0)
        check("Fold cumsum (carries across ranks)", bool((np.isnan(cs) == np.isnan(wcs)).all()) and
              bool((np.isnan(wcs) | (np.abs(cs - wcs) <= 4 * math.log2(n) * EPS * run_abs + 1e-300)).all()))
        check("Fold cummax", exact(P(dv.cummax()).to_numpy(), vals.cummax().to_numpy()))
        check("Fold ffill", exact(P(dv.ffill()).to_numpy(), vals.ffill().to_numpy()))
        # Reduce: var / std, two packed all-reduces
        check("Reduce var", bool(np.allclose(np.asarray(P(dv.var())), vals.var().to_numpy(), rtol=16 * math.log2(n) * EPS, atol=0)))
        check("Reduce std(ddof=0)", bool(np.allclose(np.asarray(P(dv.std(ddof=0))), vals.std(ddof=0).to_numpy(),
                                                     rtol=16 * math.log2(n) * EPS, atol=0)))
        spec = {"c1": "mean", "c0": "sum"}
        ga, wa = P(df.groupby("key").agg(spec)), pdf.groupby("key").agg(spec)
        check("groupby.agg(dict)", list(ga.index) == list(wa.index) and list(ga.columns) == list(wa.columns) and
              bool(np.allclose(ga.to_numpy(), wa.to_numpy(), rtol=0, atol=1e-9, equal_nan=True)))
        check("reduction of a reduction stays local", bool(np.isclose(float((dv.sum() * 2.0).sum()), (vals.sum() * 2.0).sum(), rtol=1e-12)))


def main():
    import argparse

    ap = argparse.ArgumentParser()
    ap.add_argument("--api", default="both", choices=["mirror", "modin", "both"])
    args = ap.parse_args()
    assert dist.init_from_env("nccl"), "run under torchrun with WORLD_SIZE > 1"
    rank, ws = dist.rank(), dist.world_size()
    config.NPartitions.put(2)
    fails = []
    apis = ["mirror", "modin"] if args.api == "both" else [args.api]
    if "modin" in apis and not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "modin")):
        apis.remove("modin")
        if rank == 0:
            print("SKIP modin front door: oracle/_ref/modin is not installed", flush=True)
    for which in apis:
        try:
            run_checks(front_door(which), which, rank, fails)
        except Exception as exc:
            import traceback

            fails.append(f"[{which}] crashed: {type(exc).__name__}: {exc}")
            if rank == 0:
                traceback.print_exc()
    t = torch.tensor([len(fails)], dtype=torch.int64, device="cuda")
    torch.distributed.all_reduce(t)
    if rank == 0:
        print(f"dist_check: {'OK' if int(t.item()) == 0 else 'FAILED'} on {ws} ranks", flush=True)
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()
    sys.exit(0 if int(t.item()) == 0 else 1)


if __name__ == "__main__":
    main()
