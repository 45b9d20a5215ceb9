"""Composite keys across row-range shards (partial-record merge, padded merge, the one-call communicator step, chunked
aggregation) against the oracle on the whole data, in global first-appearance order.  Shards agree on one key layout
(distributed.agree_layouts over every shard's GroupBy.key_layout()) and repack to it before the local pass; the owners
merge the packed words and unpack them.  Needs a GPU: -m gpu."""
import numpy as np
import pyarrow as pa
import pytest

from test_distributed_composite_cpu import pack_model

pytestmark = pytest.mark.gpu

ALL = ["sum", "mean", "count", "min", "max", "first", "last"]
KEYS = ["k1", "k2"]


@pytest.fixture(scope="module")
def pab():
    import pandasarrow_b200 as p
    return p


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


class Data:
    """Config-3-shaped columns: k1 int32, k2 dictionary<int32 -> utf8> over ONE dictionary shared by every shard,
    1 % null keys; nullable fp64 / int64 / boolean values.  `clean` lists, per shard, the key columns that carry no
    validity bitmap on that shard (so that the shards' own layouts differ)."""

    def __init__(self, n, n1, nsym, seed, world=1, clean=()):
        rng = np.random.default_rng(seed)
        self.n, self.world = n, world
        self.k1 = rng.integers(0, n1, n).astype(np.int32)
        self.k2 = rng.integers(0, nsym, n).astype(np.int32)
        self.m1, self.m2 = rng.random(n) < 0.01, rng.random(n) < 0.01
        self.dictionary = pa.array([f"sym{i:03d}" for i in range(nsym)])
        from pandasarrow_b200 import distributed as D
        self.shards = [D.shard_rows(n, world, r) for r in range(world)]
        for r, cols in enumerate(clean):
            b, e = self.shards[r]
            if "k1" in cols:
                self.m1[b:e] = False
            if "k2" in cols:
                self.m2[b:e] = False
        self.clean = list(clean) + [()] * (world - len(clean))
        i = rng.integers(-50, 50, n)
        vm = rng.random(n) < 0.1
        self.vals = {"f": pa.array(rng.random(n) * 100 - 30, pa.float64(), mask=vm), "i": pa.array(i, pa.int64(), mask=vm),
                     "b": pa.array(rng.random(n) < 0.7, pa.bool_(), mask=vm)}

    def keys(self, b, e, clean=()):
        m1 = None if "k1" in clean else self.m1[b:e]
        m2 = None if "k2" in clean else self.m2[b:e]
        return (pa.array(self.k1[b:e], pa.int32(), mask=m1),
                pa.DictionaryArray.from_arrays(pa.array(self.k2[b:e], pa.int32(), mask=m2), self.dictionary))

    def batch(self):
        k1, k2 = self.keys(0, self.n)
        return pa.record_batch({"k1": k1, "k2": k2, **self.vals})

    def shard_handle(self, pab, r, **kw):
        b, e = self.shards[r]
        k1, k2 = self.keys(b, e, self.clean[r])
        frame = {"k1": k1, "k2": k2, **{c: v.slice(b, e - b) for c, v in self.vals.items()}}
        return pab.GroupBy(KEYS, frame, row_base=b, **kw), frame


def _agree(handles):
    from pandasarrow_b200 import distributed as D
    agreed = D.agree_layouts([g.key_layout() for g in handles])
    for g in handles:
        g.set_key_layout(agreed)
    return agreed


def _merge(pab, handles, frames, world, aggs, col, agreed, dictionaries):
    """Emulated ranks on one GPU: every shard exports its records (and distinct pairs) by owner; owner o merges the o-th
    segment of every source in source order, as the NCCL all-to-all delivers them.  Returns [k1, k2], {agg: array}."""
    import torch
    from pandasarrow_b200 import distributed as D
    from pandasarrow_b200._lib import PA_AGG, PA_AGG_STAGE2, PA_DISTINCT_PAIR_WORDS as PW, PA_PARTIAL_WORDS, PA_PARTIAL_WORDS_STAGE2
    stage2 = any(PA_AGG[a] & PA_AGG_STAGE2 for a in aggs)
    W = PA_PARTIAL_WORDS_STAGE2 if stage2 else PA_PARTIAL_WORDS
    distinct = "count_distinct" in aggs
    sends, counts, psends, pcounts = [], [], [], []
    for g, fr in zip(handles, frames):
        g.aggregate(fr[col], aggs, fetch=False)
        c = g.partials_count(world)
        buf = torch.empty((max(sum(c), 1), W), dtype=torch.int64, device="cuda")
        g.partials_export(world, buf.data_ptr(), buf.shape[0], stage2=stage2)
        sends.append(buf[:sum(c)]); counts.append(c)
        if distinct:
            pc = g.distinct_pairs_count(world)
            pbuf = torch.empty((max(sum(pc), 1), PW), dtype=torch.int64, device="cuda")
            g.distinct_pairs_export(world, pbuf.data_ptr(), pbuf.shape[0])
            psends.append(pbuf[:sum(pc)]); pcounts.append(pc)

    def segments(bufs, cnts, o, words):
        segs, rc = [], []
        for s in range(len(bufs)):
            off = sum(cnts[s][:o])
            segs.append(bufs[s][off:off + cnts[s][o]]); rc.append(cnts[s][o])
        recv = torch.cat(segs).contiguous() if sum(rc) else torch.empty((1, words), dtype=torch.int64, device="cuda")
        return recv, rc

    vfmt = {pa.float64(): "g", pa.int64(): "l", pa.bool_(): "b"}[frames[0][col].type]
    out, keys, firsts = {a: [] for a in aggs}, [[], []], []
    for o in range(world):
        recv, rc = segments(sends, counts, o, W)
        m = pab.MergedGroupBy(recv.data_ptr(), rc, [a for a in aggs if a != "count_distinct"], vfmt, "L")
        m.set_composite_key(agreed, ["i", "i"], KEYS, dictionaries)
        if distinct:
            precv, prc = segments(psends, pcounts, o, PW)
            m.merge_distinct_pairs(precv.data_ptr(), prc)
        for a in aggs:
            out[a].append(m.fetch(a))
        u1, u2 = m.unique(0), m.unique(1)
        dict2 = isinstance(u2, pa.DictionaryArray)
        if len(u1):   # the owner of every merged group is the owner of its agreed packed word
            w = pack_model([u1.fill_null(0).to_numpy(), (u2.indices if dict2 else u2).fill_null(0).to_numpy()],
                           [np.asarray(u1.is_null()), np.asarray(u2.is_null())], agreed)
            assert (D.owner_of(w, world) == o).all()
        keys[0].append(u1); keys[1].append(u2.cast(pa.string()) if dict2 else u2)
        firsts.append(m.first_rows().to_numpy())
        m.close()
    order = pa.array(np.argsort(np.concatenate(firsts), kind="stable"))
    return [pa.concat_arrays(k).take(order) for k in keys], {a: pa.concat_arrays(out[a]).take(order) for a in aggs}


def _moment2(rb, col):
    import pyarrow.compute as pc
    from oracle import oracle as orc
    x = rb.column(col).cast(pa.float64())
    o2 = orc.OracleGroupBy(pa.record_batch({"k1": rb.column("k1"), "k2": rb.column("k2"), "sq": pc.multiply(x, x)}), KEYS)
    m = o2.agg("mean", "sq", nthreads=8).to_numpy(zero_copy_only=False).astype(np.float64)
    o2.close()
    return np.where(np.isfinite(m), m, 0.0)


def check_oracle(orc, rb, keys, res, col, what):
    """keys: [k1, k2 as strings]; results against the oracle on the whole batch, group order = first appearance."""
    from test_stage2_gpu import _numeric
    from util import abs_scale, align_to, assert_exact, assert_fp_close, first_appearance_order, with_abs
    ours = list(zip(keys[0].to_pylist(), keys[1].to_pylist()))
    assert ours == first_appearance_order([rb.column("k1"), rb.column("k2")]), f"{what}: global first-appearance order"
    ora = orc.OracleGroupBy(with_abs(rb), KEYS)
    theirs = list(zip(ora.unique(0).to_pylist(), ora.unique(1).to_pylist()))
    perm = pa.array(align_to(ours, theirs))
    for a, got in res.items():
        got = got.take(perm)
        if a in ("all", "any"):
            want, valid = ora.agg(a, col, nthreads=8, with_validity=True)
            assert got.is_valid().to_pylist() == valid.to_pylist(), f"{what} {a} validity"
            assert got.fill_null(False).to_pylist() == want.to_pylist(), f"{what} {a}"
        elif a == "mean":
            assert_fp_close(got, _numeric(ora, "mean", col), f"{what} mean", abs_scale(ora, col, mean=True))
        elif a == "sum" and col == "f":
            assert_fp_close(got, ora.agg("sum", col, nthreads=8), f"{what} sum", abs_scale(ora, col))
        elif a in ("variance", "stddev"):
            m2 = _moment2(rb, col)
            assert_fp_close(got, _numeric(ora, a, col), f"{what} {a}", m2 if a == "variance" else np.sqrt(m2))
        else:
            assert_exact(got, ora.agg(a, col, nthreads=8), f"{what} {a}({col})")
    ora.close()


FAMILIES = [("f", ALL), ("i", ALL), ("i", ["mean", "count", "product", "variance", "stddev"]), ("b", ["all", "any", "count"]),
            ("i", ["count_distinct", "count"])]


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("n,n1,nsym,kw", [
    (60_000, 5, 8, {}),                                  # tens of groups
    (200_000, 100, 64, {}),                              # ~6 400 groups
    (400_000, 2400, 64, {"expected_groups": 150_000}),   # ~140 000 groups
])
def test_sharded_composite_matches_oracle(pab, orc, world, n, n1, nsym, kw):
    # shard 0: no null k1; shard 1 (with 4+ shards): no null key at all; the rest: nulls in both
    clean = [("k1",)] + ([("k1", "k2")] if world > 2 else [])
    d = Data(n, n1, nsym, seed=n1 + world, world=world, clean=clean)
    rb = d.batch()
    for col, aggs in FAMILIES:
        pairs = [d.shard_handle(pab, r, **kw) for r in range(world)]
        handles, frames = [p[0] for p in pairs], [p[1] for p in pairs]
        own = {tuple(g.key_layout().nullable[:2]) for g in handles}
        assert len(own) > 1, "the shards' own layouts differ"
        agreed = _agree(handles)
        assert list(agreed.nullable[:2]) == [1, 1] and list(agreed.bits[:2]) == [32, max(1, (nsym - 1).bit_length())]
        assert {tuple(g.key_layout().nullable[:2]) for g in handles} == {(1, 1)}
        keys, res = _merge(pab, handles, frames, world, aggs, col, agreed, [None, d.dictionary])
        check_oracle(orc, rb, keys, res, col, f"P={world} n1={n1} {col} {aggs[0]}")
        for g in handles:
            g.close()


@pytest.mark.parametrize("world", [2, 4])
def test_full_width_int32_pair(pab, orc, world):
    """Two non-null int32 columns use all 64 bits (no null bits), negative values and the all-ones word included."""
    from pandasarrow_b200 import distributed as D
    rng = np.random.default_rng(world)
    n = 120_000
    a = rng.choice(np.array([-1, 0, 1, -2**31, 2**31 - 1, 77, -77], np.int32), n)
    b = rng.integers(-2**31, 2**31, n, dtype=np.int64).astype(np.int32) % 997 - 498
    b[rng.random(n) < 0.05] = -1
    f = pa.array(rng.random(n))
    rb = pa.record_batch({"k1": pa.array(a), "k2": pa.array(b.astype(np.int32)), "f": f})
    handles, frames = [], []
    for r in range(world):
        s, e = D.shard_rows(n, world, r)
        fr = {"k1": pa.array(a[s:e]), "k2": pa.array(b[s:e].astype(np.int32)), "f": f.slice(s, e - s)}
        handles.append(pab.GroupBy(KEYS, fr, row_base=s)); frames.append(fr)
    agreed = _agree(handles)
    assert list(agreed.bits[:2]) == [32, 32] and list(agreed.nullable[:2]) == [0, 0]
    keys, res = _merge(pab, handles, frames, world, ALL, "f", agreed, [None, None])
    from util import align_to, assert_exact, first_appearance_order
    ours = list(zip(keys[0].to_pylist(), keys[1].to_pylist()))
    assert ours == first_appearance_order([rb.column("k1"), rb.column("k2")])
    assert (-1, -1) in ours
    ora = orc.OracleGroupBy(rb, KEYS)
    perm = pa.array(align_to(ours, list(zip(ora.unique(0).to_pylist(), ora.unique(1).to_pylist()))))
    for a in ("count", "min", "max", "first", "last"):
        assert_exact(res[a].take(perm), ora.agg(a, "f", nthreads=8), a)
    ora.close()
    for g in handles:
        g.close()


def test_padded_exchange_composite(pab, orc):
    """Few groups: the padded blocks and the single-CTA merge; then more groups than one CTA merges (4 sources of
    ~1 500 groups into one owner), where the pending merge completes through the general merge and keeps the key."""
    import torch
    for n1, world, owners in ((6, 4, 4), (190, 4, 1)):
        d = Data(100_000, n1, 8, seed=n1, world=world, clean=[("k1",)])
        if owners == 1:   # disjoint k1 per shard: ~1 700 groups per shard, ~6 900 in the merge
            for r, (b, e) in enumerate(d.shards):
                d.k1[b:e] += r * 1000
        rb = d.batch()
        pairs = [d.shard_handle(pab, r) for r in range(world)]
        handles, frames = [p[0] for p in pairs], [p[1] for p in pairs]
        agreed = _agree(handles)
        cap = 2048
        blocks = []
        for g, fr in zip(handles, frames):
            g.aggregate(fr["f"], ALL, fetch=False, wait=False)
            buf = torch.empty((owners, cap + 1, 11), dtype=torch.int64, device="cuda")
            g.partials_export_padded(owners, buf.data_ptr(), cap)
            blocks.append(buf)
        keys, out, firsts = [[], []], {a: [] for a in ALL}, []
        for o in range(owners):
            recv = torch.stack([b[o] for b in blocks]).contiguous()
            m = pab.MergedGroupBy(recv.data_ptr(), [0] * world, ALL, "g", "L", padded_block_records=cap)
            m.set_composite_key(agreed, ["i", "i"], KEYS, [None, d.dictionary])
            for a in ALL:
                out[a].append(m.fetch(a))
            keys[0].append(m.unique(0)); keys[1].append(m.unique(1).cast(pa.string()))
            firsts.append(m.first_rows().to_numpy())
            m._keep = recv
            m.close()
        order = pa.array(np.argsort(np.concatenate(firsts), kind="stable"))
        check_oracle(orc, rb, [pa.concat_arrays(k).take(order) for k in keys],
                     {a: pa.concat_arrays(v).take(order) for a, v in out.items()}, "f", f"padded n1={n1}")
        for g in handles:
            g.close()


@pytest.fixture(scope="module")
def single_rank_comm(tmp_path_factory):
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


@pytest.mark.parametrize("col,aggs", FAMILIES)
def test_communicator_step_composite(pab, orc, single_rank_comm, col, aggs):
    """pa_groupby_sharded_aggregate on a composite key: the layout gather runs, the merged handle unpacks the key with
    gb's names and dictionaries; a second step on the same handle gives the same result."""
    d = Data(300_007, 700, 64, seed=len(aggs))
    rb = d.batch()
    gb = pab.GroupBy(KEYS, rb, row_base=5_000_000_000)
    for _ in range(2):
        m = single_rank_comm.sharded_aggregate(gb, rb.column(col), aggs)
        info = single_rank_comm.key_layout_info()
        assert info["agree_ms"] > 0 and info["repack_ms"] == 0
        u2 = m.unique(1)
        assert isinstance(u2, pa.DictionaryArray) and u2.dictionary.equals(d.dictionary) and m.key_names == KEYS
        check_oracle(orc, rb, [m.unique(0), u2.cast(pa.string())], {a: m.fetch(a) for a in aggs}, col, f"comm {col} {aggs[0]}")
        m.close()
    # a single-key step runs no agreement
    g1 = pab.GroupBy("k1", rb)
    single_rank_comm.sharded_aggregate(g1, rb.column("f"), ["sum"]).close()
    assert single_rank_comm.key_layout_info() == {"agree_ms": 0.0, "repack_ms": 0.0}
    g1.close(); gb.close()


@pytest.mark.parametrize("n,chunk", [(1_000_003, 100_000), (250_000, 1 << 30), (500_001, 7_813)])
def test_chunked_composite_equals_single_gpu(pab, n, chunk):
    from util import assert_exact, assert_fp_close
    rng = np.random.default_rng(n)
    k1 = pa.array(rng.integers(0, 300, n).astype(np.int32), mask=rng.random(n) < 0.01)
    words = np.array([f"w{i}" for i in range(40)])
    k2 = pa.array(words[rng.integers(0, 40, n)], mask=rng.random(n) < 0.01)      # utf8: encoded once by the helper
    k3 = pa.DictionaryArray.from_arrays(pa.array(rng.integers(0, 5, n).astype(np.int32)),   # no nulls: no null bit
                                        pa.array([10, 20, 30, 40, 50], pa.int64()))
    v = pa.array(rng.random(n) * 10, mask=rng.random(n) < 0.1)
    aggs = ALL + ["variance", "stddev"]
    single = pab.GroupBy(["k1", "k2", "k3"], {"k1": k1, "k2": k2, "k3": k3})
    want = single.aggregate(v, aggs)
    m = pab.aggregate_chunked([k1, k2, k3], v, aggs, chunk)
    try:
        for j in range(3):
            got, exp = m.unique(j), single.unique(j)
            assert got.equals(exp), j
        for a in aggs:
            (assert_fp_close if a in ("sum", "mean", "variance", "stddev") else assert_exact)(m.fetch(a), want[a], a)
    finally:
        m.close(); single.close()


def test_set_key_layout_keeps_results(pab):
    """A local handle gives identical unique / aggregates / row ids before and after a repack to a wider layout."""
    d = Data(200_000, 50, 16, seed=3, world=1, clean=[("k1",)])
    gb, fr = d.shard_handle(pab, 0)
    own = gb.key_layout()
    assert list(own.nullable[:2]) == [0, 1] and own.dict_fingerprint[0] == 0 and own.dict_fingerprint[1] != 0
    before = (gb.unique(0), gb.unique(1), gb.aggregate(fr["f"], ALL), gb.row_ids())
    wider = gb.key_layout()
    wider.nullable[0] = 1
    gb.set_key_layout(wider)
    assert list(gb.key_layout().nullable[:2]) == [1, 1]
    after = (gb.unique(0), gb.unique(1), gb.aggregate(fr["f"], ALL), gb.row_ids())
    assert before[0].equals(after[0]) and before[1].equals(after[1]) and before[3].equals(after[3])
    for a in ALL:
        assert before[2][a].equals(after[2][a]), a
    gb.set_key_layout(wider)                                  # equal layout: no-op, the results stay fetchable
    assert gb.fetch("sum").equals(before[2]["sum"])
    gb.close()


def test_composite_errors(pab):
    from pandasarrow_b200 import distributed as D
    rng = np.random.default_rng(9)
    n = 10_000
    # each shard fits 64 bits alone, the agreed layout needs 65: int32 + two 15-bit dictionaries, nulls on different columns
    dct = pa.array(np.arange(1 << 15, dtype=np.int64))
    idx = rng.integers(0, 1 << 15, n).astype(np.int32)
    k1 = rng.integers(0, 9, n).astype(np.int32)
    nm = rng.random(n) < 0.1
    a = pab.GroupBy(["a", "b", "c"], {"a": pa.array(k1, mask=nm), "b": pa.DictionaryArray.from_arrays(pa.array(idx, mask=nm), dct),
                                      "c": pa.DictionaryArray.from_arrays(pa.array(idx), dct)})
    b = pab.GroupBy(["a", "b", "c"], {"a": pa.array(k1), "b": pa.DictionaryArray.from_arrays(pa.array(idx), dct),
                                      "c": pa.DictionaryArray.from_arrays(pa.array(idx, mask=nm), dct)})
    with pytest.raises(pab.PaError, match="needs 65 bits"):
        D.agree_layouts([a.key_layout(), b.key_layout()])
    a.close(); b.close()
    # shards encoded against different dictionaries: per-shard encoding, and same length in another order
    s = np.array(["x", "y", "z"])[rng.integers(0, 3, n)]
    s[:10] = ["x", "y", "z", "x", "y", "z", "x", "y", "z", "x"]
    v = pa.array(s)
    p0 = pab.GroupBy(KEYS, {"k1": pa.array(k1[:5000]), "k2": v.slice(0, 5000).dictionary_encode()})
    p1 = pab.GroupBy(KEYS, {"k1": pa.array(k1[5000:]), "k2": pa.array(np.where(s[5000:] == "x", "x", "y")[::-1]).dictionary_encode()})
    fwd = pa.DictionaryArray.from_arrays(pa.array([0, 1, 2], pa.int32()), pa.array(["p", "q", "r"]))
    rev = pa.DictionaryArray.from_arrays(pa.array([0, 1, 2], pa.int32()), pa.array(["q", "p", "r"]))
    q0 = pab.GroupBy(KEYS, {"k1": pa.array(k1[:3]), "k2": fwd})
    q1 = pab.GroupBy(KEYS, {"k1": pa.array(k1[:3]), "k2": rev})
    for x, y in ((p0, p1), (q0, q1)):
        with pytest.raises(pab.PaError, match="one dictionary shared by all shards"):
            D.agree_layouts([x.key_layout(), y.key_layout()])
        with pytest.raises(pab.PaError, match="dictionary"):
            y.set_key_layout(x.key_layout())
    # a narrower layout (no null bit for a column with nulls)
    g = pab.GroupBy(KEYS, {"k1": pa.array(k1, mask=nm), "k2": pa.DictionaryArray.from_arrays(pa.array(idx % 3), fwd.dictionary)})
    narrow = g.key_layout()
    narrow.nullable[0] = 0
    with pytest.raises(pab.PaError, match="has nulls"):
        g.set_key_layout(narrow)
    # a merged key must be the packed word
    import torch
    rec = torch.zeros((1, 11), dtype=torch.int64, device="cuda")
    m = pab.MergedGroupBy(rec.data_ptr(), [0], ["count"], "g", "l")
    with pytest.raises(pab.PaError, match="packed word"):
        m.set_composite_key(g.key_layout(), ["i", "i"])
    # layouts describe composite keys only; a utf8 single key is still refused across shards
    u = pab.GroupBy("s", {"s": v})
    with pytest.raises(pab.PaError, match="composite key"):
        u.key_layout()
    u.aggregate(pa.array(np.ones(n)), ["sum"], fetch=False)
    with pytest.raises(pab.PaError, match="utf8 keys"):
        u.partials_count(2)
    for h in (p0, p1, q0, q1, g, m, u):
        h.close()
