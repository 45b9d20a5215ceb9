"""A single utf8 / large_utf8 key across row-range shards (partial records with their key bytes, the one-call
communicator step, chunked aggregation) against the oracle on the whole data, in global first-appearance order.  Every
shard hashes with one agreed seed and exports its records with their key lengths and bytes; owner o merges the o-th
segment of every source and checks the bytes (pa_merge_key_strings).  The collision hook (PA_TEST_STR_HASH_BITS) is read
once per process, so those cases run in a child process.  Needs a GPU: -m gpu."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pyarrow as pa
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALL = ["sum", "mean", "count", "min", "max", "first", "last"]
FAMILIES = [("f", ALL), ("i", ["mean", "count", "product", "variance", "stddev"]), ("b", ["all", "any", "count"]),
            ("i", ["count_distinct", "count"])]
SPECIAL = ["", "ü", "日本語", "a" * 40, "ä" * 17]


@pytest.fixture(scope="module")
def pab():
    import pandasarrow_b200 as p
    return p


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


def symbols(nsym):
    return SPECIAL + [f"key{i}" + ("ß" if i % 3 == 0 else "") for i in range(nsym)]


class Data:
    """String keys (with nulls, the empty string and non-ASCII bytes) drawn per shard: `mode` "overlap" (every shard from
    all symbols), "disjoint" (shard r from its own symbols) or "identical" (every shard holds every symbol).  `empty` /
    `all_null`: shards that hold no rows / only null keys.  Nullable fp64 / int64 / boolean values."""

    def __init__(self, n, nsym, world, mode="overlap", seed=0, large=False, empty=(), all_null=(), null_p=0.02):
        rng = np.random.default_rng(seed)
        from pandasarrow_b200 import distributed as D
        sym = symbols(nsym)
        sizes = [0 if r in empty else 1 for r in range(world)]
        live = [r for r in range(world) if sizes[r]]
        bounds = [D.shard_rows(n, len(live), i) for i in range(len(live))]
        self.shards, k, i = [], 0, 0
        for r in range(world):
            if r in empty:
                self.shards.append((k, k))
                continue
            b, e = bounds[i]
            i += 1
            self.shards.append((b, e))
            k = e
        keys = np.empty(n, dtype=object)
        for r, (b, e) in enumerate(self.shards):
            if e == b:
                continue
            pool = sym if mode != "disjoint" else sym[r::world]
            if mode == "identical":
                keys[b:e] = [pool[j % len(pool)] for j in range(e - b)]
                keys[b:e] = keys[b:e][rng.permutation(e - b)]
            else:
                keys[b:e] = [pool[j] for j in rng.integers(0, len(pool), e - b)]
        nulls = rng.random(n) < null_p
        for r in all_null:
            b, e = self.shards[r]
            nulls[b:e] = True
        keys[nulls] = None
        self.n, self.world = n, world
        self.key = pa.array(list(keys), pa.large_string() if large else pa.string())
        vm = rng.random(n) < 0.1
        self.vals = {"f": pa.array(rng.random(n) * 100 - 30, pa.float64(), mask=vm),
                     "i": pa.array(rng.integers(-50, 50, n), pa.int64(), mask=vm),
                     "b": pa.array(rng.random(n) < 0.7, pa.bool_(), mask=vm)}

    def batch(self):
        return pa.record_batch({"k": self.key, **self.vals})

    def shard_handle(self, pab, r, **kw):
        b, e = self.shards[r]
        frame = {"k": self.key.slice(b, e - b), **{c: v.slice(b, e - b) for c, v in self.vals.items()}}
        return pab.GroupBy("k", frame, row_base=b, **kw), frame


def _segments(bufs, cnts, o, dtype, words=None):
    import torch
    segs, rc = [], []
    for s in range(len(bufs)):
        off = sum(cnts[s][:o])
        segs.append(bufs[s][off:off + cnts[s][o]]); rc.append(cnts[s][o])
    if sum(rc):
        return torch.cat(segs).contiguous(), rc
    return torch.empty((1, words) if words else (1,), dtype=dtype, device="cuda"), rc


def export_all(handles, frames, world, aggs, col):
    """Every shard's local pass and its records / lengths / bytes (and distinct pairs) grouped by owner."""
    import torch
    from pandasarrow_b200._lib import PA_AGG, PA_AGG_STAGE2, PA_DISTINCT_PAIR_WORDS as PW, PA_PARTIAL_WORDS, PA_PARTIAL_WORDS_STAGE2
    stage2 = any(PA_AGG[a] & PA_AGG_STAGE2 for a in aggs)
    W = PA_PARTIAL_WORDS_STAGE2 if stage2 else PA_PARTIAL_WORDS
    ex = {"W": W, "recs": [], "counts": [], "lens": [], "bytes": [], "nbytes": [], "pairs": [], "pcounts": [], "seeds": []}
    for g, fr in zip(handles, frames):
        g.aggregate(fr[col], aggs, fetch=False)
        c, b = g.partials_count_utf8(world)
        buf = torch.empty((max(sum(c), 1), W), dtype=torch.int64, device="cuda")
        lens = torch.empty(max(sum(c), 1), dtype=torch.int32, device="cuda")
        data = torch.empty(max(sum(b), 1), dtype=torch.uint8, device="cuda")
        g.partials_export_utf8(world, buf.data_ptr(), buf.shape[0], lens.data_ptr(), data.data_ptr(), data.numel(), stage2=stage2)
        ex["recs"].append(buf[:sum(c)]); ex["counts"].append(c)
        ex["lens"].append(lens[:sum(c)]); ex["bytes"].append(data[:sum(b)]); ex["nbytes"].append(b)
        ex["seeds"].append(g.key_hash_seed())
        if "count_distinct" in aggs:
            pc = g.distinct_pairs_count(world)
            pbuf = torch.empty((max(sum(pc), 1), PW), dtype=torch.int64, device="cuda")
            g.distinct_pairs_export(world, pbuf.data_ptr(), pbuf.shape[0])
            ex["pairs"].append(pbuf[:sum(pc)]); ex["pcounts"].append(pc)
    return ex


def merge_owner(pab, ex, o, aggs, vfmt, kfmt, seeds=None):
    """Owner o's merged handle and whether its byte check saw a collision."""
    import torch
    from pandasarrow_b200._lib import PA_DISTINCT_PAIR_WORDS as PW
    recv, rc = _segments(ex["recs"], ex["counts"], o, torch.int64, ex["W"])
    rlen, _ = _segments(ex["lens"], ex["counts"], o, torch.int32)
    rbytes, rbc = _segments(ex["bytes"], ex["nbytes"], o, torch.uint8)
    m = pab.MergedGroupBy(recv.data_ptr(), rc, [a for a in aggs if a != "count_distinct"], vfmt, kfmt)
    collided = m.merge_key_strings(rlen.data_ptr(), rbytes.data_ptr(), rc, rbc, seeds or ex["seeds"])
    if "count_distinct" in aggs and not collided:
        precv, prc = _segments(ex["pairs"], ex["pcounts"], o, torch.int64, PW)
        m.merge_distinct_pairs(precv.data_ptr(), prc)
    m._keep = (recv, rlen, rbytes)
    return m, collided


def merge_all(pab, handles, frames, world, aggs, col, large):
    """Emulated ranks on one GPU; returns the keys and {agg: array} in global first-appearance order."""
    ex = export_all(handles, frames, world, aggs, col)
    assert len(set(ex["seeds"])) == 1
    vfmt = {pa.float64(): "g", pa.int64(): "l", pa.bool_(): "b"}[frames[0][col].type]
    keys, out, firsts = [], {a: [] for a in aggs}, []
    for o in range(world):
        m, collided = merge_owner(pab, ex, o, aggs, vfmt, "U" if large else "u")
        assert not collided
        for a in aggs:
            out[a].append(m.fetch(a))
        keys.append(m.unique())
        firsts.append(m.first_rows().to_numpy())
        m.close()
    order = pa.array(np.argsort(np.concatenate(firsts), kind="stable"))
    return pa.concat_arrays(keys).take(order), {a: pa.concat_arrays(v).take(order) for a, v in out.items()}


def check_oracle(orc, rb, key, res, col, what):
    from test_stage2_gpu import _numeric
    from util import abs_scale, align_to, assert_exact, assert_fp_close, first_appearance_order, with_abs
    assert key.type == rb.column("k").type, f"{what}: unique() type {key.type}"
    ours = [(k,) for k in key.to_pylist()]
    assert ours == first_appearance_order([rb.column("k")]), f"{what}: global first-appearance order"
    ora = orc.OracleGroupBy(with_abs(rb), "k")
    perm = pa.array(align_to(ours, [(k,) for k in ora.unique().to_pylist()]))
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
            x = rb.column(col).cast(pa.float64()).to_numpy(zero_copy_only=False)
            sq = pa.array(x * x, mask=np.asarray(rb.column(col).is_null()))
            o2 = orc.OracleGroupBy(pa.record_batch({"k": rb.column("k"), "sq": sq}), "k")
            m2 = o2.agg("mean", "sq", nthreads=8).to_numpy(zero_copy_only=False).astype(np.float64)
            o2.close()
            m2 = np.where(np.isfinite(m2), m2, 0.0)
            assert_fp_close(got, _numeric(ora, a, col), f"{what} {a}", m2 if a == "variance" else np.sqrt(m2))
        else:
            assert_exact(got, ora.agg(a, col, nthreads=8), f"{what} {a}({col})")
    ora.close()


@pytest.mark.parametrize("world", [1, 2, 3, 4])
@pytest.mark.parametrize("mode", ["overlap", "disjoint", "identical"])
@pytest.mark.parametrize("large", [False, True])
def test_sharded_strings_match_oracle(pab, orc, world, mode, large):
    d = Data(120_000, 300, world, mode=mode, seed=world, large=large)
    rb = d.batch()
    for col, aggs in FAMILIES:
        pairs = [d.shard_handle(pab, r) for r in range(world)]
        key, res = merge_all(pab, [p[0] for p in pairs], [p[1] for p in pairs], world, aggs, col, large)
        check_oracle(orc, rb, key, res, col, f"P={world} {mode} large={large} {col} {aggs[0]}")
        for g, _ in pairs:
            g.close()


@pytest.mark.parametrize("world", [3, 4])
def test_empty_and_all_null_shards(pab, orc, world):
    d = Data(50_000, 40, world, seed=7, empty=(1,), all_null=(world - 1,))
    rb = d.batch()
    for col, aggs in FAMILIES:
        pairs = [d.shard_handle(pab, r) for r in range(world)]
        key, res = merge_all(pab, [p[0] for p in pairs], [p[1] for p in pairs], world, aggs, col, False)
        check_oracle(orc, rb, key, res, col, f"P={world} empty / all-null {col} {aggs[0]}")
        for g, _ in pairs:
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


@pytest.mark.parametrize("large", [False, True])
@pytest.mark.parametrize("col,aggs", FAMILIES)
def test_communicator_step_strings(pab, orc, single_rank_comm, large, col, aggs):
    """pa_groupby_sharded_aggregate on a utf8 key: one attempt at seed 0, every key byte sent to the one owner; a second
    step on the same handle gives the same result."""
    d = Data(200_003, 900, 1, seed=len(aggs), large=large)
    rb = d.batch()
    gb = pab.GroupBy("k", rb, row_base=3_000_000_000)
    for _ in range(2):
        m = single_rank_comm.sharded_aggregate(gb, rb.column(col), aggs)
        info = single_rank_comm.key_strings_info()
        assert info["seed"] == 0 and info["attempts"] == 1
        assert info["bytes_sent"] == info["bytes_received"] > 0
        check_oracle(orc, rb, m.unique(), {a: m.fetch(a) for a in aggs}, col, f"comm {col} {aggs[0]}")
        m.close()
    gb.close()


def test_communicator_step_unordered_export(pab, orc, single_rank_comm):
    """Millions of distinct strings, no null key, sum / mean / count of floats: after the first step (which checks the
    grouping byte for byte on the ordered groups) the step hands over the bucketed path's unordered records, and their
    key bytes follow them."""
    n = 6_000_000
    rng = np.random.default_rng(11)
    words = pa.array([f"w{i:07d}" for i in rng.permutation(3_000_000)])
    keys = pa.DictionaryArray.from_arrays(pa.array(rng.integers(0, len(words), n).astype(np.int32)), words).cast(pa.string())
    rb = pa.record_batch({"k": keys, "f": pa.array(rng.random(n))})
    gb = pab.GroupBy("k", rb, row_base=0)
    seen = []
    for _ in range(2):
        m = single_rank_comm.sharded_aggregate(gb, rb.column("f"), ["sum", "mean", "count"])
        seen.append(single_rank_comm.exchange_info()["unordered_export"])
        check_oracle(orc, rb, m.unique(), {a: m.fetch(a) for a in ("sum", "mean", "count")}, "f", "unordered export")
        m.close()
    assert seen[-1], f"unordered export not taken: {seen}"
    gb.close()


@pytest.mark.parametrize("chunk_rows", [7_001, 40_000, 1 << 20])
@pytest.mark.parametrize("large", [False, True])
def test_chunked_strings(pab, orc, chunk_rows, large):
    d = Data(150_000, 500, 1, seed=chunk_rows % 97, large=large)
    rb = d.batch()
    for col, aggs in FAMILIES[:3]:
        m = pab.aggregate_chunked(rb.column("k"), rb.column(col), aggs, chunk_rows)
        check_oracle(orc, rb, m.unique(), {a: m.fetch(a) for a in aggs}, col, f"chunked {chunk_rows} {col} {aggs[0]}")
        m.close()


def test_errors(pab):
    import torch
    d = Data(20_000, 30, 2, seed=3)
    g, fr = d.shard_handle(pab, 0)
    g.aggregate(fr["f"], ["sum"], fetch=False)
    for call in (lambda: g.partials_count(2), lambda: g.partials_export_padded(2, 1, 16)):
        with pytest.raises(pab.PaError, match="utf8 keys"):
            call()
    # the _utf8 export needs its own count first
    with pytest.raises(pab.PaError, match="partials_count_utf8"):
        g.partials_export_utf8(2, 1, 1, 1, 1, 1)
    # seeds belong to utf8 keys only
    n = pab.GroupBy("i", {"i": pa.array(np.arange(10))})
    n.aggregate(pa.array(np.ones(10)), ["sum"], fetch=False)
    with pytest.raises(pab.PaError, match="utf8"):
        n.key_hash_seed()
    with pytest.raises(pab.PaError, match="utf8"):
        n.partials_count_utf8(2)
    rec = torch.zeros((1, 11), dtype=torch.int64, device="cuda")
    with pytest.raises(pab.PaError, match="counted exchange"):
        pab.MergedGroupBy(rec.data_ptr(), [0, 0], ["sum"], "g", "u", padded_block_records=4)
    # unique() and distinct pairs before the key strings are attached
    ex = export_all([g], [fr], 1, ["count_distinct", "count"], "i")
    m = pab.MergedGroupBy(ex["recs"][0].data_ptr(), ex["counts"][0], ["count"], "l", "u")
    with pytest.raises(pab.PaError, match="pa_merge_key_strings"):
        m.unique()
    with pytest.raises(pab.PaError, match="pa_merge_key_strings"):
        m.merge_distinct_pairs(ex["pairs"][0].data_ptr(), ex["pcounts"][0])
    # differing seeds are refused
    with pytest.raises(pab.PaError, match="different seeds"):
        m.merge_key_strings(ex["lens"][0].data_ptr(), ex["bytes"][0].data_ptr(), ex["counts"][0] + [0], ex["nbytes"][0] + [0], [0, 1])
    assert not m.merge_key_strings(ex["lens"][0].data_ptr(), ex["bytes"][0].data_ptr(), ex["counts"][0], ex["nbytes"][0], [0])
    assert m.unique().to_pylist() == g.unique().to_pylist()
    for h in (g, n, m):
        h.close()


HOOK = textwrap.dedent(r'''
    import sys
    sys.path[:0] = [{root!r}, {tests!r}]
    import numpy as np
    import pyarrow as pa
    import pandasarrow_b200 as pab
    from test_sharded_strkeys_gpu import export_all, merge_owner

    def shard(keys, b):
        fr = {{"k": pa.array(keys), "f": pa.array(np.arange(len(keys), dtype=np.float64) + b)}}
        return pab.GroupBy("k", fr, row_base=b), fr

    # across shards only: shard 0 holds "a", shard 1 holds "b"; under seed 0 (every hash bit dropped) they share a hash
    hs = [shard(["a", "a", "a"], 0), shard(["b", "b"], 3)]
    ex = export_all([h for h, _ in hs], [f for _, f in hs], 1, ["sum", "count"], "f")
    assert ex["seeds"] == [0, 0], ex["seeds"]
    m, collided = merge_owner(pab, ex, 0, ["sum", "count"], "g", "u")
    assert collided, "cross-shard collision not seen"
    m.close()
    for h, _ in hs:
        h.set_key_hash_seed(1)
    ex = export_all([h for h, _ in hs], [f for _, f in hs], 1, ["sum", "count"], "f")
    m, collided = merge_owner(pab, ex, 0, ["sum", "count"], "g", "u")
    assert not collided
    assert m.unique().to_pylist() == ["a", "b"] and m.fetch("sum").to_pylist() == [3.0, 7.0], m.fetch("sum")
    m.close()

    # inside one shard: its own check moves it to seed 1; the owner refuses until the seeds are agreed
    hs = [shard(["a", "b", "a"], 0), shard(["b", "b"], 3)]
    ex = export_all([h for h, _ in hs], [f for _, f in hs], 1, ["count"], "f")
    assert ex["seeds"] == [1, 0], ex["seeds"]
    try:
        merge_owner(pab, ex, 0, ["count"], "g", "u")
        raise SystemExit("differing seeds accepted")
    except pab.PaError as e:
        assert "different seeds" in str(e)
    hs[1][0].set_key_hash_seed(1)
    ex = export_all([h for h, _ in hs], [f for _, f in hs], 1, ["count"], "f")
    m, collided = merge_owner(pab, ex, 0, ["count"], "g", "u")
    assert not collided and m.unique().to_pylist() == ["a", "b"] and m.fetch("count").to_pylist() == [2, 3]
    m.close()

    # chunked: chunk 0 = "a"..., chunk 1 = "b"...: the merge sees the collision and the chunks are redone with seed 1
    k = pa.array(["a"] * 5 + ["b"] * 5, pa.large_string())
    m = pab.aggregate_chunked(k, pa.array(np.arange(10.0)), ["sum", "count"], 5)
    assert m.unique().type == pa.large_string() and m.unique().to_pylist() == ["a", "b"]
    assert m.fetch("sum").to_pylist() == [10.0, 35.0] and m.fetch("count").to_pylist() == [5, 5]
    m.close()
    print("HOOK OK")
''')


def test_collision_hook():
    """PA_TEST_STR_HASH_BITS=0 makes every hash under seed 0 equal: a collision across shards only (seen by the owner), one
    inside a shard (its own check moves the seed) and one across chunks, each ending in the oracle's groups."""
    env = dict(os.environ, PA_TEST_STR_HASH_BITS="0")
    code = HOOK.format(root=ROOT, tests=os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    print(r.stdout[-4000:], r.stderr[-4000:])
    assert r.returncode == 0 and "HOOK OK" in r.stdout
