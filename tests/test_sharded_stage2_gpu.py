"""Product / variance / stddev across row-range shards (multi-GPU step, partial-record merge, chunked aggregation)
against the oracle on the whole data.  Every shard runs the two-pass second stage on its own rows and ships its terms
(M2 around its own mean, its product) in PA_PARTIAL_WORDS_STAGE2-word records; the owner combines them in source-rank
order (Chan's update for M2, a plain product).  Needs a GPU: -m gpu.

Bars as in test_stage2_gpu.py: variance / stddev within 1e-12 relative to max(value, mean(x^2)) resp. its square root;
integer products bit-exact (wrapping); float products within 1e-12 relative."""
import numpy as np
import pyarrow as pa
import pytest

from test_stage2_gpu import _frame, _numeric, _second_moment

pytestmark = pytest.mark.gpu

S2 = ["product", "variance", "stddev"]
ALL = ["sum", "mean", "count", "min", "max", "first", "last"]
FMT = {pa.float64(): "g", pa.float32(): "f", pa.int64(): "l", pa.int32(): "i", pa.uint16(): "S"}


@pytest.fixture(scope="module")
def pab():
    import pandasarrow_b200 as p
    return p


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


def _merge_shards(pab, shards, world, aggs, vfmt, kfmt, make_handle):
    """Emulated ranks on one GPU: shard r (a (begin, end) row range) is aggregated by make_handle(r) -> (handle, value
    column) and exported as stage-2 records; owner o merges the o-th segment of every source's records, in source
    order (what the NCCL all-to-all delivers).  Returns keys, {agg: array}, first rows — global first-row order."""
    import torch
    from pandasarrow_b200 import distributed as D
    from pandasarrow_b200._lib import PA_PARTIAL_WORDS_STAGE2 as W
    sends, counts = [], []
    for r in range(len(shards)):
        g, col = make_handle(r)
        g.aggregate(col, aggs, fetch=False)
        c = g.partials_count(world)
        buf = torch.empty((max(sum(c), 1), W), dtype=torch.int64, device="cuda")
        g.partials_export(world, buf.data_ptr(), buf.shape[0], stage2=True)
        sends.append(buf[:sum(c)]); counts.append(c)
        g.close()
    out = {a: [] for a in aggs}
    keys, firsts = [], []
    for o in range(world):
        segs, rc = [], []
        for s in range(len(shards)):
            off = sum(counts[s][:o])
            segs.append(sends[s][off:off + counts[s][o]]); rc.append(counts[s][o])
        recv = torch.cat(segs).contiguous() if sum(rc) else torch.empty((1, W), dtype=torch.int64, device="cuda")
        m = pab.MergedGroupBy(recv.data_ptr(), rc, aggs, vfmt, kfmt)
        for a in aggs:
            out[a].append(m.fetch(a))
        k = m.unique()
        if len(k):
            own = D.owner_of(k.fill_null(0).to_numpy().astype(np.int64), world, is_null=np.asarray(k.is_null()))
            assert (own == o).all()
        keys.append(k); firsts.append(m.first_rows().to_numpy())
        m.close()
    fr = np.concatenate(firsts)
    order = pa.array(np.argsort(fr, kind="stable"))
    return pa.concat_arrays(keys).take(order), {a: pa.concat_arrays(out[a]).take(order) for a in aggs}, np.sort(fr)


def _run_sharded(pab, rb, col, aggs, world, shards=None, **kw):
    from pandasarrow_b200 import distributed as D
    n = rb.num_rows
    shards = shards or [D.shard_rows(n, world, r) for r in range(world)]

    def make(r):
        b, e = shards[r]
        shard = rb.slice(b, e - b)
        return pab.GroupBy("k", shard, row_base=b, **kw), shard.column(col)
    return _merge_shards(pab, shards, world, aggs, FMT[rb.column(col).type], "l", make)


def _check_against_oracle(orc, rb, keys, res, col, what, check_var=True, check_prod=True):
    from util import align_to, assert_exact, assert_fp_close, first_appearance_order
    ours = [(x,) for x in keys.to_pylist()]
    assert ours == first_appearance_order([rb.column("k")]), f"{what}: global first-appearance order"
    ora = orc.OracleGroupBy(rb, "k")
    perm = pa.array(align_to(ours, [(x,) for x in ora.unique().to_pylist()]))
    if "count" in res:
        assert_exact(res["count"].take(perm), ora.agg("count", col, nthreads=8), f"{what} count({col})")
    if check_var:
        m2 = _second_moment(rb, ora, col)
        assert_fp_close(res["variance"].take(perm), _numeric(ora, "variance", col), f"{what} variance({col})", m2)
        assert_fp_close(res["stddev"].take(perm), _numeric(ora, "stddev", col), f"{what} stddev({col})", np.sqrt(m2))
        if "mean" in res:
            assert_fp_close(res["mean"].take(perm), _numeric(ora, "mean", col), f"{what} mean({col})", np.sqrt(m2))
    if check_prod:
        got, want = res["product"].take(perm), ora.agg("product", col, nthreads=8)
        (assert_fp_close if pa.types.is_floating(rb.column(col).type) else assert_exact)(got, want, f"{what} product({col})")
    ora.close()


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("n,G,kw", [
    (60_000, 5, {}),                                   # warp-combined updates on every shard
    (200_000, 300, {}),                                # CTA-shared accumulators
    (300_000, 20_000, {}),                             # L2 atomics
    (300_000, 150_000, {"expected_groups": 150_000}),
])
def test_sharded_stage2_matches_oracle(pab, orc, world, n, G, kw):
    rb = _frame(n, G, seed=G + world)
    aggs = ["mean", "count"] + S2
    for col in ("f", "w", "w32", "i", "i32", "u16"):
        keys, res, fr = _run_sharded(pab, rb, col, aggs, world, **kw)
        assert len(np.unique(fr)) == len(fr)
        # products of the normal(3, 2) columns leave the normal range: their variance is what they are here for
        _check_against_oracle(orc, rb, keys, res, col, f"P={world} G={G}", check_prod=col not in ("w", "w32"))


def _edge_frame():
    """Three row-range shards built so that groups meet the merge's corner cases (key: what it tests)."""
    nan, inf = float("nan"), float("inf")
    shards = [
        [(1, 1.0), (1, 2.0), (3, None), (4, 2.5), (5, 1.0), (6, 2.0), (8, 1.0), (9, 1e6 + 1), (9, 1e6 - 1), (9, 1e6 + 0.5)],
        [(1, None), (1, None), (2, 4.0), (2, 6.0), (2, 8.0), (4, 2.5), (4, 2.5), (5, nan), (5, 2.0), (8, 3.0),
         (9, -1e6 + 2), (9, -1e6 - 2), (10, -inf), (None, 5.0), (11, 1e6 + 7), (11, 1e6 + 9)],
        [(3, None), (4, 2.5), (5, 3.0), (6, inf), (6, 1.0), (7, 7.0), (9, 1e6 + 3), (10, 3.0), (None, 1.0),
         (11, -1e6), (11, -1e6 + 4)],
    ]
    # 1: valid in shard 0, all-null in shard 1        2: in shard 1 only         3: all-null everywhere
    # 4: constant, split over all shards              5: NaN in one shard        6: +inf in one shard
    # 7: a single row                                 8: single rows in two shards
    # 9, 11: shards whose means are ~2e6 apart        10: -inf in one shard      null key: split over two shards
    bounds, rows, b = [], [], 0
    for s in shards:
        rows += s
        bounds.append((b, b + len(s)))
        b += len(s)
    rb = pa.record_batch({"k": pa.array([r[0] for r in rows], pa.int64()), "v": pa.array([r[1] for r in rows], pa.float64())})
    return rb, bounds


@pytest.mark.parametrize("world", [1, 3])
def test_sharded_stage2_edge_cases(pab, orc, world):
    rb, bounds = _edge_frame()
    aggs = ["count", "mean"] + S2
    keys, res, _ = _run_sharded(pab, rb, "v", aggs, world, shards=bounds)
    _check_against_oracle(orc, rb, keys, res, "v", f"edge P={world}")
    assert keys.to_pylist() == [1, 3, 4, 5, 6, 8, 9, 2, 10, None, 11, 7]
    got = {k: {a: res[a][i].as_py() for a in aggs} for i, k in enumerate(keys.to_pylist())}
    assert got[1]["variance"] == 0.25 and got[1]["product"] == 2.0 and got[1]["count"] == 2
    assert got[2]["variance"] == pytest.approx(8 / 3, rel=1e-15) and got[2]["product"] == 192.0
    assert got[3] == {"count": 0, "mean": None, "product": None, "variance": None, "stddev": None}
    assert got[4]["variance"] == 0.0 and got[4]["stddev"] == 0.0 and got[4]["product"] == 2.5 ** 4
    assert np.isnan(got[5]["variance"]) and np.isnan(got[5]["product"])
    assert np.isnan(got[6]["variance"]) and got[6]["product"] == float("inf")
    assert np.isnan(got[10]["variance"]) and got[10]["product"] == float("-inf")
    assert got[7]["variance"] == 0.0 and got[7]["product"] == 7.0
    assert got[8]["variance"] == 1.0 and got[8]["product"] == 3.0
    assert got[None]["variance"] == 4.0 and got[None]["product"] == 5.0
    for k, vals in ((9, [1e6 + 1, 1e6 - 1, 1e6 + 0.5, -1e6 + 2, -1e6 - 2, 1e6 + 3]), (11, [1e6 + 7, 1e6 + 9, -1e6, -1e6 + 4])):
        x = np.array(vals)
        want = np.mean((x - x.mean()) ** 2)
        assert abs(got[k]["variance"] - want) <= 1e-12 * max(want, np.mean(x * x)), k
    # integer products that wrap, the factors of one group spread over the shards
    ib = pa.record_batch({"k": pa.array([0] * 70 + [1] * 3 + [0] * 10, pa.int64()),
                          "v": pa.array([3] * 70 + [-7, 11, 13] + [5] * 10, pa.int64())})
    keys, res, _ = _run_sharded(pab, ib, "v", ["product", "variance"], world, shards=[(0, 30), (30, 72), (72, 83)])
    whole = pab.GroupBy("k", ib)
    assert res["product"].equals(whole.product("v"))
    assert res["product"].equals(orc.OracleGroupBy(ib, "k").agg("product", "v"))
    assert res["product"].to_pylist()[1] == -1001
    whole.close()


def test_stage2_records_errors(pab):
    import torch
    from pandasarrow_b200._lib import PA_PARTIAL_WORDS_STAGE2 as W
    rb = pa.record_batch({"k": pa.array([1, 2, 1, 3], pa.int64()), "v": pa.array([1.0, 2.0, 3.0, 4.0])})
    g = pab.GroupBy("k", rb)
    buf = torch.empty((8, W), dtype=torch.int64, device="cuda")
    # no second stage in the last aggregate: nothing to export
    g.aggregate(rb.column("v"), ["sum", "count"], fetch=False)
    c = g.partials_count(1)
    with pytest.raises(pab.PaError, match="no product / variance / stddev"):
        g.partials_export(1, buf.data_ptr(), buf.shape[0], stage2=True)
    # ... also after a stage-2 aggregate was superseded by an ordinary one
    g.aggregate(rb.column("v"), ["variance"], fetch=False)
    g.aggregate(rb.column("v"), ["sum"], fetch=False)
    c = g.partials_count(1)
    with pytest.raises(pab.PaError, match="no product / variance / stddev"):
        g.partials_export(1, buf.data_ptr(), buf.shape[0], stage2=True)
    # records of a product-only aggregate carry no variance terms
    g.aggregate(rb.column("v"), ["product"], fetch=False)
    c = g.partials_count(1)
    g.partials_export(1, buf.data_ptr(), buf.shape[0], stage2=True)
    m = pab.MergedGroupBy(buf.data_ptr(), c, ["product", "count"], "g", "l")
    assert m.fetch("product").to_pylist() == [3.0, 2.0, 4.0]
    with pytest.raises(pab.PaError, match="no variance / product terms"):
        pab.MergedGroupBy(buf.data_ptr(), c, ["variance"], "g", "l")
    # the padded (single-CTA) merge stays PA_AGG_ALL-only
    blocks = torch.zeros((1, 9, 11), dtype=torch.int64, device="cuda")
    with pytest.raises(pab.PaError, match="bad aggregate mask"):
        pab.MergedGroupBy(blocks.data_ptr(), [0], ["variance"], "g", "l", padded_block_records=8)
    # count_distinct / all / any stay refused on the sharded paths
    with pytest.raises(pab.PaError, match="bad aggregate mask"):
        pab.MergedGroupBy(buf.data_ptr(), c, ["count_distinct"], "g", "l")
    with pytest.raises(pab.PaError, match="chunked aggregates"):
        pab.aggregate_chunked(rb.column("k"), rb.column("v"), ["count_distinct"], 2)
    g.close()


@pytest.fixture(scope="module")
def single_rank_comm(tmp_path_factory):
    """A pa_comm of world size 1 over a one-process gloo group (as in test_multigpu_gpu.py)."""
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


@pytest.mark.parametrize("aggs", [["mean", "variance", "stddev", "product"], ALL + ["variance"]], ids=["stage2", "all+variance"])
@pytest.mark.parametrize("G,nulls,vtype", [(700, False, "f64"), (40_000, True, "f64"), (3000, True, "i64")])
def test_communicator_step_stage2_records(pab, orc, single_rank_comm, aggs, G, nulls, vtype):
    """pa_groupby_sharded_aggregate with stage-2 bits: 104-byte records, never the compact or unordered export;
    results against the oracle with global row numbers beyond 32 bits; a narrow step on the same handle afterwards
    travels as before."""
    from util import abs_scale, align_to, assert_exact, assert_fp_close, first_appearance_order, with_abs
    rng = np.random.default_rng(G + len(aggs))
    n = 300_007
    k = pa.array(rng.integers(-G // 2, G // 2, n), pa.int64(), mask=(rng.random(n) < 0.01) if nulls else None)
    vmask = (rng.random(n) < 0.05) if nulls else None
    if vtype == "i64":
        v = pa.array(rng.choice([-3, -2, -1, 1, 2, 3], n), pa.int64(), mask=vmask)   # (no zero factor: products wrap)
    else:
        v = pa.array(np.where(rng.random(n) < 0.3, -1.0, 1.0) * np.exp(rng.normal(0.0, 0.05, n)), mask=vmask)
    rb = pa.record_batch({"k": k, "v": v})
    row_base = 5_000_000_000
    gb = pab.GroupBy("k", rb, row_base=row_base)
    m = single_rank_comm.sharded_aggregate(gb, rb.column("v"), aggs)
    info = single_rank_comm.exchange_info()
    assert info == {"record_bytes": 104, "unordered_export": False, "merge_table_slots": info["merge_table_slots"]}
    ora = orc.OracleGroupBy(with_abs(rb), "k")
    ours = [(x,) for x in m.unique().to_pylist()]
    assert ours == first_appearance_order([rb.column("k")]), "global first-appearance order"
    perm = pa.array(align_to(ours, [(x,) for x in ora.unique().to_pylist()]))
    fr = m.first_rows().to_numpy()
    assert (np.diff(fr) > 0).all() and fr[0] == row_base
    m2 = _second_moment(rb, ora, "v")
    for a in aggs:
        got = m.fetch(a).take(perm)
        if a in ("variance", "stddev"):
            assert_fp_close(got, _numeric(ora, a, "v"), a, m2 if a == "variance" else np.sqrt(m2))
        elif a == "mean":
            assert_fp_close(got, _numeric(ora, "mean", "v"), a, abs_scale(ora, "v", mean=True))
        elif (a == "sum" or a == "product") and vtype != "i64":
            assert_fp_close(got, ora.agg(a, "v", nthreads=8), a, abs_scale(ora, "v") if a == "sum" else None)
        else:
            assert_exact(got, ora.agg(a, "v", nthreads=8), a)
    m.close()
    m = single_rank_comm.sharded_aggregate(gb, rb.column("v"), ["sum", "mean", "count"])
    assert single_rank_comm.exchange_info()["record_bytes"] == (88 if vtype == "i64" else 32)
    m.close(); gb.close(); ora.close()


@pytest.mark.parametrize("n,chunk,G", [(1_000_003, 100_000, 500), (1_000_003, 333_334, 40_000), (250_000, 1 << 30, 1000), (700_001, 11_000, 3)])
def test_chunked_stage2_of_host_columns(pab, orc, n, chunk, G):
    """pa_groupby_aggregate_chunked with product / variance / stddev: every chunk's terms travel in stage-2 records and
    are merged in chunk (= row) order — against the oracle on the whole columns, group order included."""
    from util import abs_scale, align_to, assert_exact, assert_fp_close, first_appearance_order, with_abs
    rng = np.random.default_rng(n + chunk)
    k = pa.array(rng.integers(-G // 2, G - G // 2, n) * 7919, pa.int64())
    v = pa.array(np.where(rng.random(n) < 0.3, -1.0, 1.0) * np.exp(rng.normal(0.0, 0.05, n)), pa.float64(), mask=rng.random(n) < 0.03)
    frame = {"k": k, "v": v}
    ora = orc.OracleGroupBy(with_abs(frame), "k")
    aggs = ALL + S2
    m = pab.aggregate_chunked(k, v, aggs, chunk)
    try:
        ours = [(x,) for x in m.unique().to_pylist()]
        assert ours == first_appearance_order([k]), "not in global first-appearance order"
        perm = pa.array(align_to(ours, [(x,) for x in ora.unique().to_pylist()]))
        m2 = _second_moment(pa.record_batch(frame), ora, "v")
        for a in aggs:
            got = m.fetch(a).take(perm)
            if a in ("variance", "stddev"):
                assert_fp_close(got, _numeric(ora, a, "v"), a, m2 if a == "variance" else np.sqrt(m2))
            elif a == "mean":
                assert_fp_close(got, _numeric(ora, "mean", "v"), a, abs_scale(ora, "v", mean=True))
            elif a == "sum":
                assert_fp_close(got, ora.agg("sum", "v", nthreads=8), a, abs_scale(ora, "v"))
            elif a == "product":
                assert_fp_close(got, ora.agg("product", "v", nthreads=8), a)
            else:
                assert_exact(got, ora.agg(a, "v", nthreads=8), a)
    finally:
        m.close()
        ora.close()


@pytest.mark.parametrize("world", [2, 5])
def test_sharded_resample_stage2_equals_single_gpu(pab, world):
    """Row-range shards of a resample with the common anchor (start of the day of the global first tick): merged
    variance / stddev / product equal the single-GPU Resampler."""
    from util import assert_fp_close
    rng = np.random.default_rng(11 + world)
    n, freq = 300_000, 7 * 60 * 10**9
    ts = np.cumsum(rng.integers(1, 3_000_000_000, n)).astype(np.int64) + 1_577_836_800_000_000_000 + 5 * 3600 * 10**9
    idx = pa.array(ts, pa.timestamp("ns"))
    v = pa.array(rng.normal(size=n) + 100.0, mask=rng.random(n) < 0.1)
    q = pa.array(rng.integers(1, 4, n), pa.int64())
    single = pab.resample({"v": v, "q": q}, idx, freq)
    want_v = single.aggregate(v, ["mean", "variance", "stddev"])
    want_q = single.aggregate(q, ["product", "variance", "mean"])
    anchor = int(ts[0] - ts[0] % (86_400 * 10**9))
    from pandasarrow_b200 import distributed as D
    shards = [D.shard_rows(n, world, r) for r in range(world)]
    scale = {}
    for col, want in (("v", want_v), ("q", want_q)):
        mean = want["mean"].to_numpy(zero_copy_only=False)
        scale[col] = np.nan_to_num(want["variance"].to_numpy(zero_copy_only=False) + mean * mean)
    for col, aggs, want in ((v, ["mean", "variance", "stddev"], want_v), (q, ["product", "variance"], want_q)):
        def make(r, col=col):
            b, e = shards[r]
            return pab.resample({"x": col.slice(b, e - b)}, idx.slice(b, e - b), freq, origin="custom",
                                origin_custom_ns=anchor, row_base=b), col.slice(b, e - b)
        labels, got, _ = _merge_shards(pab, shards, world, aggs, "g" if col is v else "l", "tsn:", make)
        assert labels.cast(pa.int64()).equals(single.index().cast(pa.int64()))
        m2 = scale["v" if col is v else "q"]
        for a in aggs:
            if a == "product":
                assert got[a].equals(want[a]), a
            else:
                assert_fp_close(got[a], want[a], f"{a} P={world}", m2 if a == "variance" else (np.sqrt(m2) if a == "stddev" else None))
    single.close()
