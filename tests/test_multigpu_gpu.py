"""Multi-GPU path (SURVEY §8e) with the ranks emulated on ONE GPU: P row-range shards are aggregated
one after the other, their partial records are routed to the owners by plain concatenation (what the
NCCL all-to-all does across GPUs), each owner merges, and the union is compared with the oracle on
the full data set.  Needs a GPU: -m gpu."""
import numpy as np
import pyarrow as pa
import pytest

pytestmark = pytest.mark.gpu

ALL = ["sum", "mean", "count", "min", "max", "first", "last"]
FMT = {pa.float64(): "g", pa.int64(): "l", pa.float32(): "f", pa.int32(): "i"}


def _run_sharded(pab, rb, key, col, aggs, world, path="auto", on_merged=None):
    import torch
    from pandasarrow_b200 import distributed as D
    from pandasarrow_b200._lib import PA_PARTIAL_WORDS as W
    n = rb.num_rows
    sends, counts = [], []
    for r in range(world):
        b, e = D.shard_rows(n, world, r)
        shard = rb.slice(b, e - b)
        g = pab.GroupBy(key, shard, row_base=b, path=path)
        g.aggregate(shard.column(col), aggs, fetch=False)
        c = g.partials_count(world)
        buf = torch.empty((max(sum(c), 1), W), dtype=torch.int64, device="cuda")
        g.partials_export(world, buf.data_ptr(), buf.shape[0])
        sends.append(buf[:sum(c)]); counts.append(c)
        g.close()
    out = {a: [] for a in aggs}
    keys, firsts = [], []
    for o in range(world):   # owner o receives, from every source s, the o-th segment of s's send buffer
        segs, rc = [], []
        for s in range(world):
            off = sum(counts[s][:o])
            segs.append(sends[s][off:off + counts[s][o]]); rc.append(counts[s][o])
        recv = torch.cat(segs).contiguous() if sum(rc) else torch.empty((1, W), dtype=torch.int64, device="cuda")
        m = pab.MergedGroupBy(recv.data_ptr(), rc, aggs, FMT[rb.column(col).type], FMT.get(rb.column(key).type, "l"))
        for a in aggs:
            out[a].append(m.fetch(a))
        keys.append(m.unique()); firsts.append(m.first_rows().to_numpy())
        # owner check: every key this rank merged hashes to it
        k = m.unique()
        if len(k):
            own = D.owner_of(k.fill_null(0).to_numpy().astype(np.int64), world, is_null=np.asarray(k.is_null()))
            assert (own == o).all()
        if on_merged is not None:
            on_merged(o, m)
        m.close()
    fr = np.concatenate(firsts)
    order = pa.array(np.argsort(fr, kind="stable"))
    res = {a: pa.concat_arrays(out[a]).take(order) for a in aggs}
    return pa.concat_arrays(keys).take(order), res, np.sort(fr)


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("G,path", [(1000, "auto"), (50_000, "auto"), (300, "global")])
def test_sharded_matches_oracle(world, G, path):
    import pandasarrow_b200 as pab
    from oracle import oracle as orc
    from pandasarrow_b200 import hostgen as hg
    from util import abs_scale, align_to, assert_exact, assert_fp_close, first_appearance_order, with_abs
    n = 400_003
    k = hg.keys(n, G)
    kmask = hg.valid_mask(n, seed=123, null_every=97)
    rb = pa.record_batch({"k": pa.array(k, mask=~kmask), "v": pa.array(hg.vals(n), mask=~hg.valid_mask(n))})
    keys, res, first_rows = _run_sharded(pab, rb, "k", "v", ALL, world, path)
    ora = orc.OracleGroupBy(with_abs(rb), "k")
    ours = [(x,) for x in keys.to_pylist()]
    assert ours == first_appearance_order([rb.column("k")]), "global first-appearance order"
    perm = pa.array(align_to(ours, [(x,) for x in ora.unique().to_pylist()]))
    for a in ALL:
        got = res[a].take(perm)
        if a == "mean":
            want, valid = ora.agg("mean", "v", nthreads=8, with_validity=True)
            want = pa.array(want.to_numpy(zero_copy_only=False), pa.float64(), mask=~np.asarray(valid.to_numpy(zero_copy_only=False), dtype=bool))
            assert_fp_close(got, want, f"mean P={world}", abs_scale(ora, "v", mean=True))
        elif a == "sum":
            assert_fp_close(got, ora.agg("sum", "v", nthreads=8), f"sum P={world}", abs_scale(ora, "v"))
        else:
            assert_exact(got, ora.agg(a, "v", nthreads=8), f"{a} P={world}")
    # invariants that also hold at full scale: counts add up, first rows are distinct
    assert sum(res["count"].to_pylist()) == int(hg.valid_mask(n).sum())
    assert len(np.unique(first_rows)) == len(first_rows)



@pytest.mark.parametrize("n,G", [(400_003, 1000), (12_000_000, 3_000_000)])
def test_bench_dump_outputs_per_rank(tmp_path, n, G):
    """bench.py --dump-outputs at N > 1: every owner writes the groups it merged as <name>_rank<r>.npy, all ranks
    together within the 64 MB on disk (the second case is sampled: ~1.5 M groups per rank); checked against numpy."""
    import importlib.util
    import os
    import pandasarrow_b200 as pab
    from pandasarrow_b200 import hostgen as hg
    spec = importlib.util.spec_from_file_location("pa_bench", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    world = 2
    k, v = hg.keys(n, G), hg.vals(n)
    rb = pa.record_batch({"k": pa.array(k), "v": pa.array(v)})
    rank_keys = {}

    def dump(o, m):
        rank_keys[o] = m.unique().to_numpy().astype(np.float64)
        bench.dump_outputs(m, str(tmp_path), o, world)

    _run_sharded(pab, rb, "k", "v", bench.AGGS, world, on_merged=dump)
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64_000_000
    cnt = np.bincount(k, minlength=G)
    s = np.bincount(k, weights=v, minlength=G)
    seen = 0
    for o in range(world):
        got = {a: np.load(tmp_path / f"{a}_rank{o}.npy") for a in ["keys"] + bench.AGGS}
        if os.path.exists(tmp_path / f"group_index_rank{o}.npy"):
            pos = np.load(tmp_path / f"group_index_rank{o}.npy").astype(np.int64)
            assert 0 < len(pos) < len(rank_keys[o]) and (np.diff(pos) > 0).all()
        else:
            pos = np.arange(len(rank_keys[o]))
            seen += len(pos)
        assert np.array_equal(got["keys"], rank_keys[o][pos])
        g = got["keys"].astype(np.int64)
        assert np.array_equal(got["count"], cnt[g].astype(np.float64))
        assert np.max(np.abs(got["sum"] - s[g]) / s[g]) <= 1e-12
        assert np.max(np.abs(got["mean"] - s[g] / cnt[g]) / (s[g] / cnt[g])) <= 1e-12
    if G == 1000:
        assert seen == np.count_nonzero(cnt)           # unsampled: the ranks' files hold every group once

def test_sharded_int_values_and_single_rank():
    import pandasarrow_b200 as pab
    rng = np.random.default_rng(4)
    n = 100_000
    rb = pa.record_batch({"k": pa.array(rng.integers(0, 77, n), pa.int64()), "v": pa.array(rng.integers(-9, 9, n), pa.int64())})
    k1, r1, _ = _run_sharded(pab, rb, "k", "v", ALL, 1)
    k3, r3, _ = _run_sharded(pab, rb, "k", "v", ALL, 3)
    whole = pab.GroupBy("k", rb)
    w = whole.aggregate(rb.column("v"), ALL)
    assert k1.equals(whole.unique()) and k3.equals(whole.unique())
    for a in ALL:
        assert r1[a].equals(w[a]) and r3[a].equals(w[a]), a     # integer / positional aggregates: bit exact across P


def _run_sharded_padded(pab, rb, key, col, aggs, world, cap):
    """Same as _run_sharded, through the padded (no host round trip) exchange: block [s][o] of rank s's
    export goes to owner o."""
    import torch
    from pandasarrow_b200 import distributed as D
    from pandasarrow_b200._lib import PA_PARTIAL_WORDS as W
    n = rb.num_rows
    sends = []
    for r in range(world):
        b, e = D.shard_rows(n, world, r)
        shard = rb.slice(b, e - b)
        g = pab.GroupBy(key, shard, row_base=b)
        g.aggregate(shard.column(col), aggs, fetch=False)
        buf = torch.empty((world, cap + 1, W), dtype=torch.int64, device="cuda")
        g.partials_export_padded(world, buf.data_ptr(), cap)
        sends.append(buf)
        g.close()
    torch.cuda.synchronize()
    out = {a: [] for a in aggs}
    keys, firsts = [], []
    for o in range(world):
        recv = torch.stack([sends[s][o] for s in range(world)]).contiguous()
        m = pab.MergedGroupBy(recv.data_ptr(), [0] * world, aggs, FMT[rb.column(col).type], FMT.get(rb.column(key).type, "l"),
                              padded_block_records=cap)
        for a in aggs:
            out[a].append(m.fetch(a))
        keys.append(m.unique()); firsts.append(m.first_rows().to_numpy())
        m.close()
    fr = np.concatenate(firsts)
    order = pa.array(np.argsort(fr, kind="stable"))
    return pa.concat_arrays(keys).take(order), {a: pa.concat_arrays(out[a]).take(order) for a in aggs}


@pytest.mark.parametrize("world", [1, 2, 8])
def test_padded_exchange_equals_counted_exchange(world):
    import pandasarrow_b200 as pab
    from pandasarrow_b200 import hostgen as hg
    n, G = 300_007, 500     # <= 640 groups: the wide aggregates stay on the deterministic shared-memory path
    kmask = hg.valid_mask(n, seed=5, null_every=89)
    rb = pa.record_batch({"k": pa.array(hg.keys(n, G), mask=~kmask), "v": pa.array(hg.vals(n), mask=~hg.valid_mask(n))})
    k1, r1, _ = _run_sharded(pab, rb, "k", "v", ALL, world)
    k2, r2 = _run_sharded_padded(pab, rb, "k", "v", ALL, world, cap=2048)
    assert k1.equals(k2)
    for a in ALL:
        assert r1[a].equals(r2[a]), a          # same records, same source-rank fold order: bit for bit


def test_padded_exchange_overflow_marker():
    import pandasarrow_b200 as pab
    from pandasarrow_b200 import hostgen as hg
    n, G = 100_000, 5000
    rb = pa.record_batch({"k": pa.array(hg.keys(n, G)), "v": pa.array(hg.vals(n))})
    with pytest.raises(pab.PaError, match="padded block"):
        _run_sharded_padded(pab, rb, "k", "v", ["sum"], 2, cap=2048)


@pytest.mark.parametrize("world", [2, 5])
@pytest.mark.parametrize("closed_right,label_right", [(False, False), (True, True)])
def test_sharded_resample_equals_single_gpu(world, closed_right, label_right):
    """SURVEY §8e last row: a sorted index sharded by row range; every shard cuts the same bucket grid (common
    custom anchor = start of the day of the GLOBAL first tick), partial buckets meet in the ordinary merge."""
    import torch
    import pandasarrow_b200 as pab
    from pandasarrow_b200 import distributed as D
    from pandasarrow_b200._lib import PA_PARTIAL_WORDS as W
    from util import assert_exact, assert_fp_close
    rng = np.random.default_rng(11)
    n, freq = 300_000, 7 * 60 * 10**9            # 7 minutes does not divide a day: the grid depends on the anchor
    ts = np.cumsum(rng.integers(1, 3_000_000_000, n)).astype(np.int64) + 1_577_836_800_000_000_000 + 5 * 3600 * 10**9
    idx = pa.array(ts, pa.timestamp("ns"))
    v = pa.array(rng.normal(size=n), mask=rng.random(n) < 0.1)
    single = pab.resample({"v": v}, idx, freq, closed_right=closed_right, label_right=label_right)
    want = single.aggregate(v, ALL)
    anchor = int(ts[0] - ts[0] % (86_400 * 10**9))
    sends, counts = [], []
    for r in range(world):
        b, e = D.shard_rows(n, world, r)
        sv = v.slice(b, e - b)
        g = pab.resample({"v": sv}, idx.slice(b, e - b), freq, closed_right=closed_right, label_right=label_right,
                         origin="custom", origin_custom_ns=anchor, row_base=b)
        g.aggregate(sv, ALL, fetch=False)
        c = g.partials_count(world)
        buf = torch.empty((max(sum(c), 1), W), dtype=torch.int64, device="cuda")
        g.partials_export(world, buf.data_ptr(), buf.shape[0])
        sends.append(buf[:sum(c)]); counts.append(c)
        g.close()
    keys, firsts, out = [], [], {a: [] for a in ALL}
    for o in range(world):
        segs, rc = [], []
        for s_ in range(world):
            off = sum(counts[s_][:o])
            segs.append(sends[s_][off:off + counts[s_][o]]); rc.append(counts[s_][o])
        recv = torch.cat(segs).contiguous() if sum(rc) else torch.empty((1, W), dtype=torch.int64, device="cuda")
        m = pab.MergedGroupBy(recv.data_ptr(), rc, ALL, "g", "tsn:")
        for a in ALL:
            out[a].append(m.fetch(a))
        keys.append(m.unique()); firsts.append(m.first_rows().to_numpy())
        m.close()
    order = pa.array(np.argsort(np.concatenate(firsts), kind="stable"))
    labels = pa.concat_arrays(keys).take(order)
    assert labels.cast(pa.int64()).equals(single.index().cast(pa.int64()))          # same buckets, time order
    for a in ALL:
        got = pa.concat_arrays(out[a]).take(order)
        (assert_fp_close if a in ("sum", "mean") else assert_exact)(got, want[a], f"{a} P={world}")


@pytest.fixture(scope="module")
def single_rank_comm(tmp_path_factory):
    """A pa_comm of world size 1 (NCCL communicator with one rank) over a one-process gloo group: the whole sharded
    step — count, export, self send/recv, merge — through pa_groupby_sharded_aggregate on a single GPU."""
    import torch.distributed as dist
    from pandasarrow_b200 import distributed as D
    own_group = not dist.is_initialized()
    if own_group:
        store = dist.FileStore(str(tmp_path_factory.mktemp("pg") / "store"), 1)
        dist.init_process_group("gloo", store=store, rank=0, world_size=1)
    comm = D.Comm(device=0)
    yield comm
    comm.close()
    if own_group:
        dist.destroy_process_group()


@pytest.mark.parametrize("aggs", [["sum", "mean", "count"], ["count"], ALL], ids=["compact", "compact-count", "full"])
@pytest.mark.parametrize("G,nulls,vtype", [(700, False, "f64"), (40_000, True, "f64"), (3000, True, "i64"), (500, False, "f32")])
def test_communicator_step_compact_and_full_records(single_rank_comm, aggs, G, nulls, vtype):
    """sum / mean-of-floats / count travel as 32-byte compact records, everything else as the full 88-byte record
    (merge.cuh); both against the oracle, with a null key group, null values and global row numbers beyond 32 bits."""
    import pandasarrow_b200 as pab
    from oracle import oracle as orc
    from util import abs_scale, align_to, assert_exact, assert_fp_close, first_appearance_order, with_abs
    rng = np.random.default_rng(G)
    n = 300_007
    k = pa.array(rng.integers(-G // 2, G // 2, n), pa.int64(), mask=(rng.random(n) < 0.01) if nulls else None)
    vmask = (rng.random(n) < 0.05) if nulls else None
    if vtype == "i64":
        v = pa.array(rng.integers(-10**6, 10**6, n), pa.int64(), mask=vmask)
    else:
        v = pa.array(rng.normal(size=n).astype(np.float32 if vtype == "f32" else np.float64), mask=vmask)
    rb = pa.record_batch({"k": k, "v": v})
    row_base = 5_000_000_000
    gb = pab.GroupBy("k", rb, row_base=row_base)
    m = single_rank_comm.sharded_aggregate(gb, rb.column("v"), aggs)
    compact = vtype != "i64" or "mean" not in aggs           # the mean of integers carries a double sum: full record
    assert single_rank_comm.exchange_info()["record_bytes"] == (32 if compact and len(aggs) <= 3 else 88)
    ora = orc.OracleGroupBy(with_abs(rb), "k")
    ours = [(x,) for x in m.unique().to_pylist()]
    assert ours == first_appearance_order([rb.column("k")]), "global first-appearance order"
    perm = pa.array(align_to(ours, [(x,) for x in ora.unique().to_pylist()]))
    fr = m.first_rows().to_numpy()
    assert (np.diff(fr) > 0).all() and fr[0] == row_base
    for a in aggs:
        got = m.fetch(a).take(perm)
        if a == "mean":
            want, valid = ora.agg("mean", "v", nthreads=8, with_validity=True)
            want = pa.array(want.to_numpy(zero_copy_only=False), pa.float64(), mask=~np.asarray(valid.to_numpy(zero_copy_only=False), dtype=bool))
            assert_fp_close(got, want, "mean", abs_scale(ora, "v", mean=True))
        elif a == "sum" and vtype != "i64":
            assert_fp_close(got, ora.agg("sum", "v", nthreads=8), "sum", abs_scale(ora, "v"))
        else:
            assert_exact(got, ora.agg(a, "v", nthreads=8), a)
    m.close(); gb.close(); ora.close()


@pytest.mark.parametrize("world", [3, 8])
def test_merge_of_disjoint_key_sets_outgrows_the_hinted_table(world):
    """The join table of a merge is sized by its largest source first (row-range shards of one column mostly share
    their keys); shards with DISJOINT key sets hold `world` times as many keys, the probe bound trips and the merge is
    redone with the table sized by the record count — same result as the single-GPU pass."""
    import pandasarrow_b200 as pab
    from oracle import oracle as orc
    from util import abs_scale, align_to, assert_exact, assert_fp_close, first_appearance_order, with_abs
    rng = np.random.default_rng(world)
    per, G = 120_000, 50_000
    k = np.concatenate([rng.integers(0, G, per) * world + r for r in range(world)]).astype(np.int64)   # shard r: keys = r mod world
    rb = pa.record_batch({"k": pa.array(k), "v": pa.array(rng.normal(size=per * world))})
    keys, res, _ = _run_sharded(pab, rb, "k", "v", ALL, world)
    ora = orc.OracleGroupBy(with_abs(rb), "k")
    ours = [(x,) for x in keys.to_pylist()]
    assert ours == first_appearance_order([rb.column("k")])
    perm = pa.array(align_to(ours, [(x,) for x in ora.unique().to_pylist()]))
    for a in ALL:
        got, want = res[a].take(perm), ora.agg(a, "v", nthreads=8)
        if a in ("sum", "mean"):
            assert_fp_close(got, want, a, abs_scale(ora, "v", mean=(a == "mean")))
        else:
            assert_exact(got, want, a)
    ora.close()


@pytest.mark.parametrize("hint", [True, False])
def test_communicator_step_exports_unordered_bucket_records(single_rank_comm, hint):
    """Millions of groups + compact records: the local pass of the sharded step leaves the bucketed path's unordered
    group records as they are and the export reads them directly (no local ordering); the merged result still comes
    out in global first-appearance order and equals the oracle.  A wide aggregate set on the same handle afterwards
    takes the ordinary ordered route."""
    import pandasarrow_b200 as pab
    from oracle import oracle as orc
    from pandasarrow_b200 import hostgen as hg
    from util import assert_exact, assert_fp_close
    n, G = 6_000_000, 3_000_000
    rb = pa.record_batch({"k": pa.array(hg.keys(n, G)), "v": pa.array(hg.vals(n))})
    row_base = 7_000_000_000
    gb = pab.GroupBy("k", rb, row_base=row_base, **({"expected_groups": G} if hint else {}))
    ora = orc.OracleGroupBy(rb, "k")
    import pandas as pd
    fa = pd.unique(rb.column("k").to_numpy())
    theirs = ora.unique().to_numpy()
    pos = pd.Series(np.arange(len(theirs)), index=theirs)
    perm = pa.array(pos.loc[fa].to_numpy())
    for aggs in (["sum", "mean", "count"], ["sum", "min", "max", "last"]):
        m = single_rank_comm.sharded_aggregate(gb, rb.column("v"), aggs)
        assert gb.timing()["mode"] == "bucketed"
        info = single_rank_comm.exchange_info()
        assert info == {"record_bytes": 32 if "mean" in aggs else 88, "unordered_export": "mean" in aggs, "merge_table_slots": info["merge_table_slots"]}
        assert np.array_equal(m.unique().to_numpy(), fa), "global first-appearance order"
        fr = m.first_rows().to_numpy()
        assert fr[0] == row_base and (np.diff(fr) > 0).all()
        for a in aggs:
            got, want = m.fetch(a), ora.agg(a, "v", nthreads=8).take(perm)
            (assert_fp_close if a in ("sum", "mean") else assert_exact)(got, want, a)
        m.close()
    gb.close(); ora.close()
