"""count_distinct, all and any across row-range shards (multi-GPU step, partial-record + distinct-pair merge, chunked
aggregation) against the oracle on the whole data, group order included.  all / any merge the records' min / max of the
0 / 1 values; count_distinct ships every shard's distinct (key, value bits) pairs to the key's owner, which counts them
without duplicates.  Needs a GPU: -m gpu."""
import numpy as np
import pyarrow as pa
import pytest

pytestmark = pytest.mark.gpu

FMT = {pa.float64(): "g", pa.float32(): "f", pa.int64(): "l", pa.int32(): "i", pa.uint16(): "S", pa.bool_(): "b"}


@pytest.fixture(scope="module")
def pab():
    import pandasarrow_b200 as p
    return p


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


def _merge_shards(pab, shards, world, aggs, vfmt, kfmt, make_handle):
    """Emulated ranks on one GPU: shard r is aggregated by make_handle(r) -> (handle, value column); its partial records
    and (with count_distinct) its distinct pairs are exported by owner; owner o merges the o-th segment of every source,
    in source order (what the NCCL all-to-all delivers).  Returns keys, {agg: array}, first rows, pairs received per
    owner — global first-row order."""
    import torch
    from pandasarrow_b200 import distributed as D
    from pandasarrow_b200._lib import PA_DISTINCT_PAIR_WORDS as PW, PA_PARTIAL_WORDS as W
    distinct = "count_distinct" in aggs
    rec_aggs = [a for a in aggs if a != "count_distinct"]
    sends, counts, psends, pcounts = [], [], [], []
    for r in range(len(shards)):
        g, col = make_handle(r)
        g.aggregate(col, aggs, fetch=False)
        c = g.partials_count(world)
        buf = torch.empty((max(sum(c), 1), W), dtype=torch.int64, device="cuda")
        g.partials_export(world, buf.data_ptr(), buf.shape[0])
        sends.append(buf[:sum(c)]); counts.append(c)
        if distinct:
            pc = g.distinct_pairs_count(world)
            pbuf = torch.empty((max(sum(pc), 1), PW), dtype=torch.int64, device="cuda")
            g.distinct_pairs_export(world, pbuf.data_ptr(), pbuf.shape[0])
            psends.append(pbuf[:sum(pc)]); pcounts.append(pc)
        g.close()

    def segments(bufs, cnts, o, words):
        segs, rc = [], []
        for s in range(len(shards)):
            off = sum(cnts[s][:o])
            segs.append(bufs[s][off:off + cnts[s][o]]); rc.append(cnts[s][o])
        recv = torch.cat(segs).contiguous() if sum(rc) else torch.empty((1, words), dtype=torch.int64, device="cuda")
        return recv, rc

    out = {a: [] for a in aggs}
    keys, firsts, received = [], [], []
    for o in range(world):
        recv, rc = segments(sends, counts, o, W)
        m = pab.MergedGroupBy(recv.data_ptr(), rc, rec_aggs, vfmt, kfmt)
        if distinct:
            precv, prc = segments(psends, pcounts, o, PW)
            m.merge_distinct_pairs(precv.data_ptr(), prc)
            received.append(sum(prc))
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
    return pa.concat_arrays(keys).take(order), {a: pa.concat_arrays(out[a]).take(order) for a in aggs}, np.sort(fr), received


def _run_sharded(pab, rb, col, aggs, world, shards=None, **kw):
    from pandasarrow_b200 import distributed as D
    n = rb.num_rows
    shards = shards or [D.shard_rows(n, world, r) for r in range(world)]

    def make(r):
        b, e = shards[r]
        shard = rb.slice(b, e - b)
        return pab.GroupBy("k", shard, row_base=b, **kw), shard.column(col)
    return _merge_shards(pab, shards, world, aggs, FMT[rb.column(col).type], "l", make)


def _oracle_perm(orc, rb, keys):
    from util import align_to, first_appearance_order
    ours = [(x,) for x in keys.to_pylist()]
    assert ours == first_appearance_order([rb.column("k")]), "global first-appearance order"
    ora = orc.OracleGroupBy(rb, "k")
    return ora, pa.array(align_to(ours, [(x,) for x in ora.unique().to_pylist()]))


def _check_bool(ora, perm, res, col, what):
    for a in ("all", "any"):
        want, valid = ora.agg(a, col, nthreads=8, with_validity=True)
        got = res[a].take(perm)
        assert got.type == pa.bool_(), what
        assert got.is_valid().to_pylist() == valid.to_pylist(), f"{what} {a} validity"
        assert got.fill_null(False).to_pylist() == want.to_pylist(), f"{what} {a}"


def _frame(n, G, seed):
    rng = np.random.default_rng(seed)
    k = rng.integers(0, G, n) * 7919 - 3
    vm = rng.random(n) < 0.1
    vm[k % 13 == 5] = True                                       # all-null groups
    i = rng.integers(-40, 40, n)
    f = i.astype(np.float64) / 4
    f[rng.random(n) < 0.01] = -0.0
    f[rng.random(n) < 0.01] = np.nan
    f[rng.random(n) < 0.005] = np.inf
    return pa.record_batch({
        "k": pa.array(k, pa.int64(), mask=rng.random(n) < 0.02),
        "f": pa.array(f, pa.float64(), mask=vm),
        "f32": pa.array(f.astype(np.float32), pa.float32(), mask=vm),
        "r": pa.array(rng.normal(size=n), pa.float64(), mask=vm),   # (almost) every value distinct
        "i": pa.array(i, pa.int64(), mask=vm), "i32": pa.array(i.astype(np.int32), pa.int32(), mask=vm),
        "u16": pa.array((i + 40).astype(np.uint16), pa.uint16(), mask=vm),
        "b": pa.array(rng.random(n) < 0.5, pa.bool_(), mask=vm)})


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("n,G,kw", [
    (60_000, 5, {}),
    (200_000, 300, {}),
    (300_000, 20_000, {}),
    (300_000, 150_000, {"expected_groups": 150_000}),
])
def test_sharded_count_distinct_matches_oracle(pab, orc, world, n, G, kw):
    rb = _frame(n, G, seed=G + world)
    for col in ("f", "f32", "r", "i", "i32", "u16", "b"):
        keys, res, fr, _ = _run_sharded(pab, rb, col, ["count_distinct", "count"], world, **kw)
        assert len(np.unique(fr)) == len(fr)
        ora, perm = _oracle_perm(orc, rb, keys)
        got = res["count_distinct"].take(perm)
        assert got.type == pa.int64() and got.null_count == 0
        assert got.equals(ora.agg("count_distinct", col, nthreads=8)), f"P={world} G={G} count_distinct({col})"
        assert res["count"].take(perm).equals(ora.agg("count", col, nthreads=8))
        ora.close()


def _bits(vals):
    return np.asarray(vals, dtype=np.float64).view(np.uint64)


def test_sharded_count_distinct_edge_cases(pab, orc):
    from pandasarrow_b200 import distributed as D
    nan1 = _bits([np.nan])[0]
    nan2 = np.array([nan1 | 1], np.uint64).view(np.float64)[0]         # another NaN payload
    nan3 = np.array([nan1 | (1 << 63)], np.uint64).view(np.float64)[0]  # negative NaN
    inf = np.inf
    shards = [
        [(1, 0.0), (1, 1.0), (2, None), (3, nan2), (4, 5.0), (None, 1.0), (6, 2.0)],
        [],                                                               # a shard with 0 rows
        [(1, -0.0), (2, None), (3, np.nan), (4, 5.0), (5, inf), (None, None), (6, None)],
        [(1, 0.0), (2, None), (3, nan3), (3, nan2), (4, 6.0), (5, -inf), (None, 1.0), (6, 2.0), (7, 7.0)],
    ]
    # 1: signed zeros over shards   2: all null everywhere   3: NaN payloads over shards   4: repeated value over shards
    # 5: +-inf                      6: all null on one shard   7: a key on a single shard   null key: over three shards
    bounds, rows, b = [], [], 0
    for s in shards:
        rows += s
        bounds.append((b, b + len(s)))
        b += len(s)
    v = np.array([0.0 if r[1] is None else r[1] for r in rows], np.float64)   # (numpy keeps the NaN payloads bit for bit)
    rb = pa.record_batch({"k": pa.array([r[0] for r in rows], pa.int64()),
                          "v": pa.array(v, pa.float64(), mask=np.array([r[1] is None for r in rows]))})
    assert len(np.unique(_bits(rb.column("v").to_numpy(zero_copy_only=False)[[3, 9, 16, 17]]))) == 3
    want = {1: 3, 2: 0, 3: 3, 4: 2, None: 1, 6: 1, 5: 2, 7: 1}
    whole = pab.GroupBy("k", rb)
    single = dict(zip(whole.unique().to_pylist(), whole.count_distinct("v").to_pylist()))
    whole.close()
    assert single == want
    for world in (1, 2, 3):
        keys, res, _, _ = _run_sharded(pab, rb, "v", ["count_distinct"], world, shards=bounds)
        assert keys.to_pylist() == [1, 2, 3, 4, None, 6, 5, 7]
        assert dict(zip(keys.to_pylist(), res["count_distinct"].to_pylist())) == want, world
    # every owner but one receives nothing
    cand = np.arange(1, 4000, dtype=np.int64)
    ks = cand[D.owner_of(cand, 4) == 2][:40]
    rng = np.random.default_rng(5)
    n = 20_000
    kb = pa.record_batch({"k": pa.array(rng.choice(ks, n), pa.int64()), "v": pa.array(rng.integers(0, 30, n), pa.int64())})
    keys, res, _, received = _run_sharded(pab, kb, "v", ["count_distinct"], 4)
    assert [r == 0 for r in received] == [True, True, False, True]
    ora, perm = _oracle_perm(orc, kb, keys)
    assert res["count_distinct"].take(perm).equals(ora.agg("count_distinct", "v", nthreads=8))
    ora.close()


@pytest.mark.parametrize("world", [2, 3, 8])
def test_sharded_all_any_matches_oracle(pab, orc, world):
    rng = np.random.default_rng(40 + world)
    n, G = 200_000, 900
    k = rng.integers(0, G, n)
    b = rng.random(n) < 0.97
    b[k % 5 == 0] = True
    b[k % 7 == 1] = False
    vm = rng.random(n) < 0.1
    vm[k % 11 == 3] = True
    rb = pa.record_batch({"k": pa.array(k, pa.int64(), mask=rng.random(n) < 0.01), "b": pa.array(b, pa.bool_(), mask=vm)})
    keys, res, _, _ = _run_sharded(pab, rb, "b", ["all", "any", "count"], world)
    ora, perm = _oracle_perm(orc, rb, keys)
    _check_bool(ora, perm, res, "b", f"P={world}")
    assert res["count"].take(perm).equals(ora.agg("count", "b", nthreads=8))
    assert len(set(res["all"].to_pylist())) == 3 and len(set(res["any"].to_pylist())) >= 2
    ora.close()
    keys, res, _, _ = _run_sharded(pab, rb, "b", ["all", "any", "count_distinct"], world)
    ora, perm = _oracle_perm(orc, rb, keys)
    _check_bool(ora, perm, res, "b", f"P={world} with count_distinct")
    assert res["count_distinct"].take(perm).equals(ora.agg("count_distinct", "b", nthreads=8))
    ora.close()


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


@pytest.mark.parametrize("G,col", [(700, "f"), (40_000, "r"), (3000, "i")])
def test_communicator_step_count_distinct(pab, orc, single_rank_comm, G, col):
    """pa_groupby_sharded_aggregate with count_distinct: full records, the pair exchange visible in distinct_info, results
    against the oracle with global row numbers beyond 32 bits; a narrow step on the same handle afterwards travels in
    32-byte records and exchanges no pairs."""
    rb = _frame(300_007, G, seed=G)
    row_base = 5_000_000_000
    gb = pab.GroupBy("k", rb, row_base=row_base)
    aggs = ["count_distinct", "mean", "count"]
    m = single_rank_comm.sharded_aggregate(gb, rb.column(col), aggs)
    assert single_rank_comm.exchange_info()["record_bytes"] == 88
    ora, perm = _oracle_perm(orc, rb, m.unique())
    got = m.fetch("count_distinct").take(perm)
    assert got.equals(ora.agg("count_distinct", col, nthreads=8))
    assert m.fetch("count").take(perm).equals(ora.agg("count", col, nthreads=8))
    fr = m.first_rows().to_numpy()
    assert (np.diff(fr) > 0).all() and fr[0] == row_base
    D_ = int(np.asarray(got).sum())
    info = single_rank_comm.distinct_info()
    slots = 1024
    while slots < 2 * D_:
        slots *= 2
    assert info == {"pairs_sent": D_, "pairs_received": D_, "set_slots": slots}
    m.close()
    m = single_rank_comm.sharded_aggregate(gb, rb.column("r"), ["sum", "mean", "count"])
    assert single_rank_comm.exchange_info()["record_bytes"] == 32
    assert single_rank_comm.distinct_info() == {"pairs_sent": 0, "pairs_received": 0, "set_slots": 0}
    m.close(); gb.close(); ora.close()


def test_communicator_step_all_any(pab, orc, single_rank_comm):
    rng = np.random.default_rng(3)
    n, G = 300_007, 2000
    k = rng.integers(0, G, n)
    b = rng.random(n) < 0.9
    b[k % 5 == 0] = True
    b[k % 7 == 1] = False
    vm = rng.random(n) < 0.1
    vm[k % 11 == 3] = True
    rb = pa.record_batch({"k": pa.array(k, pa.int64(), mask=rng.random(n) < 0.01), "b": pa.array(b, pa.bool_(), mask=vm)})
    gb = pab.GroupBy("k", rb, row_base=1 << 33)
    m = single_rank_comm.sharded_aggregate(gb, rb.column("b"), ["all", "any", "count"])
    assert single_rank_comm.exchange_info()["record_bytes"] == 88
    ora, perm = _oracle_perm(orc, rb, m.unique())
    _check_bool(ora, perm, {a: m.fetch(a) for a in ("all", "any")}, "b", "comm step")
    assert len(set(m.fetch("all").to_pylist())) == 3
    with pytest.raises(pab.PaError, match="not part of the last"):
        m.fetch("min")
    m.close(); gb.close(); ora.close()


@pytest.mark.parametrize("n,chunk", [(1_000_003, 100_000), (640_000, 10_000), (250_000, 1 << 30), (500_001, 7_813)])
def test_chunked_all_any_of_host_columns(pab, orc, n, chunk):
    rng = np.random.default_rng(n + chunk)
    G = 3000
    k = rng.integers(0, G, n)
    b = rng.random(n) < 0.98
    b[k % 5 == 0] = True
    b[k % 7 == 1] = False
    vm = rng.random(n) < 0.05
    vm[k % 11 == 3] = True
    kk, bb = pa.array(k * 31, pa.int64()), pa.array(b, pa.bool_(), mask=vm)
    rb = pa.record_batch({"k": kk, "b": bb})
    m = pab.aggregate_chunked(kk, bb, ["all", "any", "count"], chunk)
    try:
        ora, perm = _oracle_perm(orc, rb, m.unique())
        _check_bool(ora, perm, {a: m.fetch(a) for a in ("all", "any")}, "b", f"chunk={chunk}")
        assert m.fetch("count").take(perm).equals(ora.agg("count", "b", nthreads=8))
        ora.close()
    finally:
        m.close()


@pytest.mark.parametrize("world", [2, 5])
def test_sharded_resample_count_distinct_equals_single_gpu(pab, world):
    rng = np.random.default_rng(21 + world)
    n, freq = 300_000, 7 * 60 * 10**9
    ts = np.cumsum(rng.integers(1, 3_000_000_000, n)).astype(np.int64) + 1_577_836_800_000_000_000 + 5 * 3600 * 10**9
    idx = pa.array(ts, pa.timestamp("ns"))
    q = pa.array(rng.integers(0, 40, n), pa.int64(), mask=rng.random(n) < 0.1)
    single = pab.resample({"q": q}, idx, freq)
    want = single.aggregate(q, ["count_distinct"])["count_distinct"]
    anchor = int(ts[0] - ts[0] % (86_400 * 10**9))
    from pandasarrow_b200 import distributed as D
    shards = [D.shard_rows(n, world, r) for r in range(world)]

    def make(r):
        b, e = shards[r]
        return pab.resample({"x": q.slice(b, e - b)}, idx.slice(b, e - b), freq, origin="custom", origin_custom_ns=anchor,
                            row_base=b), q.slice(b, e - b)
    labels, got, _, _ = _merge_shards(pab, shards, world, ["count_distinct"], "l", "tsn:", make)
    assert labels.cast(pa.int64()).equals(single.index().cast(pa.int64()))
    assert got["count_distinct"].equals(want)
    single.close()


def test_distinct_pairs_errors(pab):
    import torch
    from pandasarrow_b200._lib import PA_DISTINCT_PAIR_WORDS as PW, PA_PARTIAL_WORDS as W
    rb = pa.record_batch({"k": pa.array([1, 2, 1, 3], pa.int64()), "v": pa.array([1.0, 2.0, 1.0, 4.0]),
                          "b": pa.array([True, False, True, None])})
    g = pab.GroupBy("k", rb)
    pbuf = torch.empty((8, PW), dtype=torch.int64, device="cuda")
    # no count_distinct in the last aggregate: no pairs
    g.aggregate(rb.column("v"), ["sum", "count"], fetch=False)
    with pytest.raises(pab.PaError, match="no count_distinct"):
        g.distinct_pairs_count(1)
    # ... also after a count_distinct aggregate was superseded by another one
    g.aggregate(rb.column("v"), ["count_distinct"], fetch=False)
    assert g.distinct_pairs_count(1) == [3]
    g.aggregate(rb.column("v"), ["sum"], fetch=False)
    with pytest.raises(pab.PaError, match="no count_distinct"):
        g.distinct_pairs_count(1)
    with pytest.raises(pab.PaError, match="no count_distinct"):
        g.distinct_pairs_export(1, pbuf.data_ptr(), pbuf.shape[0])
    # the pair merge needs a merged handle
    with pytest.raises(pab.PaError, match="pa_merge_create"):
        pab.MergedGroupBy.merge_distinct_pairs(g, pbuf.data_ptr(), [0])
    # a pair whose key no record carried
    g.aggregate(rb.column("v"), ["count_distinct", "count"], fetch=False)
    c = g.partials_count(1)
    rec = torch.empty((8, W), dtype=torch.int64, device="cuda")
    g.partials_export(1, rec.data_ptr(), rec.shape[0])
    pc = g.distinct_pairs_count(1)
    g.distinct_pairs_export(1, pbuf.data_ptr(), pbuf.shape[0])
    m = pab.MergedGroupBy(rec.data_ptr(), c, ["count"], "g", "l")
    m.merge_distinct_pairs(pbuf.data_ptr(), pc)
    assert m.fetch("count_distinct").to_pylist() == [1, 1, 1]
    m.merge_distinct_pairs(pbuf.data_ptr(), [0])                       # a second call replaces the first
    assert m.fetch("count_distinct").to_pylist() == [0, 0, 0]
    bad = pbuf[:1].clone()
    bad[0, 0] = 99
    with pytest.raises(pab.PaError, match="no merged record"):
        m.merge_distinct_pairs(bad.data_ptr(), [1])
    # count_distinct is not a record aggregate; all / any need a boolean value format
    with pytest.raises(pab.PaError, match="bad aggregate mask"):
        pab.MergedGroupBy(rec.data_ptr(), c, ["count_distinct"], "g", "l")
    with pytest.raises(pab.PaError, match="boolean column"):
        pab.MergedGroupBy(rec.data_ptr(), c, ["all"], "g", "l")
    # the padded (single-CTA) merge stays PA_AGG_ALL-only
    blocks = torch.zeros((1, 9, 11), dtype=torch.int64, device="cuda")
    for a in ("all", "any"):
        with pytest.raises(pab.PaError, match="bad aggregate mask"):
            pab.MergedGroupBy(blocks.data_ptr(), [0], [a], "b", "l", padded_block_records=8)
    m.close(); g.close()
