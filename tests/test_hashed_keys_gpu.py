"""Composite keys that do not pack into 64 bits (two int64 ids, an id with a timestamp, three or four wide columns) and
composite keys with utf8 members (encode_utf8=False): the key word is a seeded 64-bit row hash (csrc/rowkeys.cuh), and
the first pass checks every row against its group's first row.  Parity against the oracle on the same key columns, in
strict first-appearance order; downstream calls against the same calls on one int64 key holding each row's tuple id;
the collision hook; the calls that refuse a hashed key because it groups on one GPU only.  Needs a GPU: -m gpu."""
import ctypes as C
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
I64_EDGES = np.array([np.iinfo(np.int64).min, np.iinfo(np.int64).max, -1, 0, 1], dtype=np.int64)
NOT_IMPLEMENTED, INVALID = 3, 1


@pytest.fixture(scope="module")
def pab():
    import pandasarrow_b200 as p
    return p


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


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


def wide_pairs(rng, n, card, nullable):
    """Two int64 key columns over `card` distinct tuples (the edge values among them), and nullable fp64 / int64 values."""
    pool1 = np.concatenate([I64_EDGES, rng.integers(np.iinfo(np.int64).min, np.iinfo(np.int64).max, card, dtype=np.int64)])[:card]
    pool2 = np.concatenate([I64_EDGES[::-1], rng.integers(np.iinfo(np.int64).min, np.iinfo(np.int64).max, card, dtype=np.int64)])[:card]
    pick = rng.integers(0, card, n)
    k1, k2 = pool1[pick], pool2[(pick * 7 + 3) % card]
    m1 = rng.random(n) < 0.03 if nullable else None
    m2 = rng.random(n) < 0.03 if nullable else None
    return pa.record_batch({"k1": pa.array(k1, mask=m1), "k2": pa.array(k2, mask=m2),
                            "v": pa.array(rng.normal(size=n), mask=rng.random(n) < 0.05),
                            "w": pa.array(rng.integers(-10**6, 10**6, n), mask=rng.random(n) < 0.05)})


def parity(pab, orc, rb, keys, what, **kw):
    from util import compare_all, with_abs
    gb = pab.GroupBy(keys, rb, **kw)
    ora = orc.OracleGroupBy(with_abs(rb), keys)
    cols = [rb.column(k) for k in keys]
    for c in ("v", "w"):
        compare_all(gb, ora, rb, c, ALL, f"{what} {c}", key_cols=cols)
    ora.close()
    return gb


@pytest.mark.parametrize("path", ["auto", "global"])
@pytest.mark.parametrize("nullable", [False, True])
@pytest.mark.parametrize("n,card", [(1, 1), (1000, 100), (1000, 100_000), (300_000, 100), (300_000, 100_000)])
def test_two_int64_keys_match_oracle(pab, orc, n, card, nullable, path):
    rb = wide_pairs(np.random.default_rng(n + card), n, card, nullable)
    gb = parity(pab, orc, rb, ["k1", "k2"], f"n={n} card={card} nulls={nullable} {path}", path=path)
    with pytest.raises(pab.PaError) as e:
        gb.key_layout()
    assert e.value.code == NOT_IMPLEMENTED
    assert gb.key_hash_seed() == 0
    gb.close()


def test_two_int64_keys_empty(pab):
    gb = pab.GroupBy(["k1", "k2"], {"k1": pa.array([], pa.int64()), "k2": pa.array([], pa.int64())})
    assert gb.groupSize() == 0
    assert gb.unique(0).to_pylist() == [] and gb.unique(1).type == pa.int64()
    assert gb.aggregate(pa.array([], pa.float64()), ["sum", "count"])["sum"].to_pylist() == []
    gb.close()


def test_three_and_four_columns(pab, orc):
    rng = np.random.default_rng(3)
    n, card = 200_000, 5000
    pick = rng.integers(0, card, n)
    a = rng.integers(-2**31, 2**31 - 1, card).astype(np.int32)[pick]
    ts = (1_600_000_000_000_000_000 + rng.integers(0, 10**15, card))[(pick * 11) % card]
    u = rng.integers(0, 2**64 - 1, card, dtype=np.uint64)[(pick * 13) % card]
    nm = rng.random(n) < 0.02
    dct = pa.array([f"name-{i}" for i in range(40)])
    d = pa.DictionaryArray.from_arrays(pa.array((pick % 40).astype(np.int32), mask=nm), dct)
    base = {"v": pa.array(rng.normal(size=n)), "w": pa.array(rng.integers(-1000, 1000, n))}
    rb3 = pa.record_batch({"a": pa.array(a), "t": pa.array(ts, pa.timestamp("ns"), mask=nm), "u": pa.array(u), **base})
    parity(pab, orc, rb3, ["a", "t", "u"], "int32 + timestamp + uint64").close()
    rb4 = pa.record_batch({"d": d, "x": pa.array(ts.astype(np.int64)), "y": pa.array(u.astype(np.int64)), **base})
    gb = parity(pab, orc, rb4, ["d", "x", "y"], "dictionary + int64 + int64")
    u0 = gb.unique(0)
    assert isinstance(u0, pa.DictionaryArray) and u0.dictionary.equals(dct)
    gb.close()
    rb5 = pa.record_batch({"a": pa.array(a), "t": pa.array(ts, pa.timestamp("ns")), "u": pa.array(u), "d": d, **base})
    parity(pab, orc, rb5, ["a", "t", "u", "d"], "four columns").close()


def _utf8(values, mask=None, typ=pa.string()):
    return pa.array([None if mask is not None and m else x for x, m in zip(values, mask if mask is not None else [False] * len(values))], typ)


def _strings(rng, n_distinct):
    # long strings that share prefixes, the empty string, short ones
    out = {"", "a", "ab"} | {f"shared-prefix-of-a-long-key/{i:05d}" for i in range(n_distinct)}
    return sorted(out)


@pytest.mark.parametrize("case", ["int64+utf8", "utf8+utf8+int32", "large_utf8", "sliced"])
def test_utf8_members_match_oracle(pab, orc, case):
    rng = np.random.default_rng(len(case))
    n, card = 120_000, 3000
    words = _strings(rng, 400)
    pick = rng.integers(0, card, n)
    s1 = [words[i % len(words)] for i in pick]
    s2 = [words[(i * 7) % len(words)] for i in pick]
    m = rng.random(n) < 0.02
    k = rng.integers(-2**62, 2**62, card)[pick]
    base = {"v": pa.array(rng.normal(size=n)), "w": pa.array(rng.integers(-1000, 1000, n))}
    if case == "int64+utf8":
        rb, keys = pa.record_batch({"k": pa.array(k), "s": _utf8(s1, m), **base}), ["k", "s"]
    elif case == "utf8+utf8+int32":
        rb = pa.record_batch({"s": _utf8(s1), "t": _utf8(s2, m), "i": pa.array((pick % 17).astype(np.int32)), **base})
        keys = ["s", "t", "i"]
    elif case == "large_utf8":
        rb, keys = pa.record_batch({"k": pa.array(k, mask=m), "s": _utf8(s1, typ=pa.large_string()), **base}), ["k", "s"]
    else:   # offset != 0 on every column
        full = pa.record_batch({"k": pa.array(np.concatenate([[5, 6, 7], k])), "s": _utf8(["x", None, ""] + s1, np.concatenate([[False, True, False], m])),
                                "v": pa.array(np.concatenate([[1.0, 2.0, 3.0], rng.normal(size=n)])),
                                "w": pa.array(np.concatenate([[1, 2, 3], rng.integers(-1000, 1000, n)]))})
        rb, keys = full.slice(3), ["k", "s"]
    gb = parity(pab, orc, rb, keys, case, encode_utf8=False)
    for j, name in enumerate(keys):
        t = rb.schema.field(name).type
        if pa.types.is_string(t) or pa.types.is_large_string(t):
            assert gb.unique(j).type == t
    gb.close()


def test_utf8_member_empty_vs_null_and_encoded_default(pab):
    s = pa.array(["", None, "", "abcdefghijXYZ", "abcdefghijXY", None, "abcdefghijXYZ"])
    k = pa.array([1, 1, 1, 2, 2, 1, 2], pa.int64())
    v = pa.array([1.0, 2.0, 3.0, 4.0, 5.0, 6.0, 7.0])
    g = pab.GroupBy(["k", "s"], {"k": k, "s": s}, encode_utf8=False)
    assert g.unique(1).to_pylist() == ["", None, "abcdefghijXYZ", "abcdefghijXY"]
    assert g.unique(0).to_pylist() == [1, 1, 2, 2]
    assert g.sum(v).to_pylist() == [4.0, 8.0, 11.0, 5.0]
    g.close()
    e = pab.GroupBy(["k", "s"], {"k": k.cast(pa.int32()), "s": s})   # default: host dictionary encoding, packed key
    assert isinstance(e.unique(1), pa.DictionaryArray) and e.key_layout().n_keys == 2
    e.close()


def test_null_slots_with_garbage_group_by_null_pattern(pab, orc):
    from util import compare_all, with_abs
    n = 50_000
    rng = np.random.default_rng(11)
    k1 = rng.integers(0, 5, n).astype(np.int64) << 40
    k2 = rng.integers(np.iinfo(np.int64).min, np.iinfo(np.int64).max, n, dtype=np.int64)   # garbage under the nulls
    k2[rng.random(n) < 0.5] = 77
    valid2 = rng.random(n) < 0.4
    valid1 = rng.random(n) < 0.8
    bits = lambda v: pa.py_buffer(np.packbits(v, bitorder="little").tobytes())
    a1 = pa.Array.from_buffers(pa.int64(), n, [bits(valid1), pa.py_buffer(k1.tobytes())])
    a2 = pa.Array.from_buffers(pa.int64(), n, [bits(valid2), pa.py_buffer(k2.tobytes())])
    rb = pa.record_batch({"k1": a1, "k2": a2, "v": pa.array(rng.normal(size=n)), "w": pa.array(rng.integers(0, 9, n))})
    gb = pab.GroupBy(["k1", "k2"], rb)
    expect = {(x if a else None, y if b else None) for x, y, a, b in zip(k1.tolist(), k2.tolist(), valid1, valid2)}
    assert gb.groupSize() == len(expect)
    ora = orc.OracleGroupBy(with_abs(rb), ["k1", "k2"])
    compare_all(gb, ora, rb, "v", ALL, "garbage nulls", key_cols=[a1, a2])
    gb.close(); ora.close()


def _tuple_ids(cols):
    seen, ids = {}, []
    for t in zip(*[c.to_pylist() for c in cols]):
        ids.append(seen.setdefault(t, len(seen)))
    return np.array(ids, dtype=np.int64)


def test_downstream_calls_match_a_tuple_id_key(pab):
    import pyarrow.compute as pc
    from util import FP_RTOL
    rng = np.random.default_rng(21)
    n, card = 200_000, 20_000
    rb = wide_pairs(rng, n, card, nullable=True)
    s = _utf8([f"member-{i % 900:04d}-with-a-long-tail" for i in rng.integers(0, 5000, n)], rng.random(n) < 0.01)
    small = pa.array(rng.choice(np.array([1, 2, -1, 1, 1, 3]), n), mask=rng.random(n) < 0.05)
    flag = pa.array(rng.random(n) < 0.7, mask=rng.random(n) < 0.05)
    for keys, cols in ((["k1", "k2"], [rb.column("k1"), rb.column("k2")]), (["k1", "s"], [rb.column("k1"), s])):
        gb = pab.GroupBy(keys, {"k1": rb.column("k1"), "k2": rb.column("k2"), "s": s}, encode_utf8=False)
        ref = pab.GroupBy("id", {"id": pa.array(_tuple_ids(cols))})
        assert gb.row_ids().equals(ref.row_ids())
        for got, want in zip(gb.groupings(), ref.groupings()):
            assert got.equals(want)
        assert gb.take_grouped(rb.column("v")).equals(ref.take_grouped(rb.column("v")))
        assert gb.first_rows().equals(ref.first_rows())
        for col, aggs in ((rb.column("v"), ["count", "min", "max", "first", "last"]),
                          (rb.column("w"), ["count", "min", "max", "first", "last", "sum", "count_distinct"]),
                          (small, ["product"]), (flag, ["all", "any"])):
            r1, r2 = gb.aggregate(col, aggs), ref.aggregate(col, aggs)
            for a in aggs:
                assert r1[a].equals(r2[a]), (keys, a)
        for a in ("sum", "mean", "variance", "stddev"):
            x = np.array(gb.aggregate(rb.column("v"), [a])[a].to_pylist(), dtype=float)
            y = np.array(ref.aggregate(rb.column("v"), [a])[a].to_pylist(), dtype=float)
            assert (np.isnan(x) == np.isnan(y)).all()
            ok = ~np.isnan(y)
            # sums of mixed-sign values compare relative to sum(|x|) of the group (the conditioning of the problem)
            scale = np.abs(y)
            if a in ("sum", "mean"):
                scale = np.maximum(scale, np.nan_to_num(np.array(ref.aggregate(pc.abs(rb.column("v")), [a])[a].to_pylist(), dtype=float)))
            assert (np.abs(x[ok] - y[ok]) <= FP_RTOL * scale[ok] + 1e-300).all(), (keys, a)
        gb.close(); ref.close()


def _device_utf8(pab, arr):
    """pa_column_to_device of a utf8 column: an ArrowDeviceArray whose offsets and bytes live on the device."""
    from pandasarrow_b200 import _lib
    from pandasarrow_b200.groupby import _CArg, _check, _Ingested, _options
    src = _CArg(arr)
    out = _lib.ArrowDeviceArray()
    opt = _options(0, "auto", 0)
    try:
        _check(_lib.load().pa_column_to_device(C.byref(src.dev), C.byref(src.schema), C.byref(opt), C.byref(out)))
        fmt = src.schema.format
    finally:
        src.close()
    assert out.array.n_buffers == 3 and out.device_type == _lib.ARROW_DEVICE_CUDA
    return out, fmt, _Ingested(out)


def test_device_resident_columns_async(pab, orc):
    import torch
    from pandasarrow_b200 import _lib
    from pandasarrow_b200.groupby import _check, _options, _pack_args
    from util import assert_fp_close, compare_all, with_abs
    rng = np.random.default_rng(31)
    rb = wide_pairs(rng, 400_000, 30_000, nullable=False)
    s = pa.array([f"device-string-{i:03d}-{'x' * (i % 13)}" for i in rng.integers(0, 300, len(rb))])
    rb = pa.record_batch({**{n: rb.column(n) for n in rb.schema.names}, "s": s})
    t1 = torch.tensor(rb.column("k1").to_numpy(), device="cuda")
    t2 = torch.tensor(rb.column("k2").to_numpy(), device="cuda")
    tv = torch.tensor(rb.column("v").fill_null(0.0).to_numpy(), device="cuda")
    L = _lib.load()
    sdev, sfmt, owner = _device_utf8(pab, s)
    args, devs, schemas = _pack_args([pab.DeviceColumn.from_torch(t1), pab.DeviceColumn.from_torch(t2), pab.DeviceColumn.from_torch(t1)])
    C.memmove(C.addressof(devs[2]), C.addressof(sdev), C.sizeof(_lib.ArrowDeviceArray))
    schemas[2].format = sfmt
    h = C.c_void_p()
    opt = _options(0, "auto", 0)
    _check(L.pa_groupby_create(devs, schemas, 3, C.byref(opt), C.byref(h)))
    gb = pab.GroupBy.__new__(pab.GroupBy)
    gb._L, gb._h, gb._frame, gb._dicts, gb.key_names, gb._key_args = L, h, {}, [None] * 3, ["k1", "k2", "s"], args
    gb._keep = (owner, t1, t2)
    dv = pab.DeviceColumn.from_torch(tv)
    host = pab.GroupBy(["k1", "k2", "s"], rb, encode_utf8=False)
    want = host.aggregate(pa.array(tv.cpu().numpy()), ["sum", "count", "min", "max"])
    abs_scale = host.aggregate(pa.array(np.abs(tv.cpu().numpy())), ["sum"])["sum"].to_numpy()
    gb.aggregate(dv, ["sum", "count", "min", "max"], fetch=False, wait=False)   # unverified: runs synchronously
    gb.aggregate(dv, ["sum", "count", "min", "max"], fetch=False, wait=False)   # verified: deferred
    for a in want:   # (floating-point sums differ in the last bits between passes: atomics order)
        if a == "sum":
            assert_fp_close(gb.fetch(a), want[a], "device-resident sum", abs_scale)
        else:
            assert gb.fetch(a).equals(want[a]), a
    for j in range(3):
        assert gb.unique(j).equals(host.unique(j))
    fr = pa.record_batch({"k1": rb.column("k1"), "k2": rb.column("k2"), "s": s, "v": pa.array(tv.cpu().numpy())})
    ora = orc.OracleGroupBy(with_abs(fr), ["k1", "k2", "s"])
    compare_all(host, ora, fr, "v", ["sum", "count", "min", "max"], "device-resident", key_cols=[fr.column(k) for k in ("k1", "k2", "s")])
    ora.close(); host.close(); gb.close()


HOOK = textwrap.dedent(r'''
    import sys
    sys.path[:0] = [{root!r}, {tests!r}]
    import numpy as np
    import pyarrow as pa
    import pandasarrow_b200 as pab
    from oracle import oracle as orc
    from util import compare_all, with_abs
    rng = np.random.default_rng(5)
    n = 20_000
    k1 = rng.integers(-2**62, 2**62, 300)[rng.integers(0, 300, n)]
    k2 = rng.integers(-2**62, 2**62, 7)[rng.integers(0, 7, n)]
    s = pa.array([("abc" * (i % 5)) + str(i % 11) for i in range(n)])
    for keys, cols in ((["k1", "k2"], {{"k1": pa.array(k1), "k2": pa.array(k2)}}), (["k1", "s"], {{"k1": pa.array(k1), "s": s}})):
        rb = pa.record_batch({{**cols, "v": pa.array(rng.normal(size=n))}})
        gb = pab.GroupBy(keys, rb, encode_utf8=False)
        ora = orc.OracleGroupBy(with_abs(rb), keys)
        compare_all(gb, ora, rb, "v", ["sum", "count", "min", "max", "first", "last"], "hook " + "+".join(keys),
                    key_cols=[rb.column(k) for k in keys])
        assert gb.key_hash_seed() == 1, gb.key_hash_seed()
        assert gb.groupSize() > 1
        gb.close(); ora.close()
    print("HOOK OK")
''')


def test_collision_hook():
    """PA_TEST_STR_HASH_BITS=0: every row hash under seed 0 is equal, the check trips and the key is re-hashed."""
    env = dict(os.environ, PA_TEST_STR_HASH_BITS="0")
    code = HOOK.format(root=ROOT, tests=os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    print(r.stdout[-4000:], r.stderr[-4000:])
    assert r.returncode == 0 and "HOOK OK" in r.stdout


def _raises(pab, code, fn, match=None):
    with pytest.raises(pab.PaError, match=match) as e:
        fn()
    assert e.value.code == code, str(e.value)


def test_refusals(pab, single_rank_comm):
    import torch
    rb = wide_pairs(np.random.default_rng(41), 10_000, 500, nullable=True)
    packed = pab.GroupBy(["k1", "k2"], {"k1": pa.array(np.arange(10_000, dtype=np.int32)), "k2": pa.array(np.arange(10_000, dtype=np.int32))})
    layout = packed.key_layout()                        # a packable composite still reports its layout
    assert layout.n_keys == 2
    gb = pab.GroupBy(["k1", "k2"], rb)
    gb.aggregate(rb.column("w"), ["sum", "count_distinct"], fetch=False)
    buf = torch.zeros(1 << 20, dtype=torch.int64, device="cuda")
    p = buf.data_ptr()
    for fn in (gb.key_layout, lambda: gb.set_key_layout(layout), lambda: gb.partials_count(2),
               lambda: gb.partials_export(2, p, 1000), lambda: gb.partials_export(2, p, 1000, stage2=True),
               lambda: gb.partials_count_utf8(2), lambda: gb.partials_export_utf8(2, p, 1000, p, p, 1000),
               lambda: gb.partials_export_padded(2, p, 100), lambda: gb.distinct_pairs_count(2),
               lambda: gb.distinct_pairs_export(2, p, 1000)):
        _raises(pab, NOT_IMPLEMENTED, fn, match="hashed composite key")
    _raises(pab, INVALID, lambda: gb.set_key_hash_seed(3))
    # the one-call step fails on every rank, and the communicator stays usable for a packed step
    _raises(pab, NOT_IMPLEMENTED, lambda: single_rank_comm.sharded_aggregate(gb, rb.column("v"), ["sum"]), match="groups on one GPU")
    v = pa.array(np.ones(10_000))
    m = single_rank_comm.sharded_aggregate(packed, v, ["sum"])
    assert m.groupSize() == 10_000 and m.fetch("sum").to_pylist()[:3] == [1.0, 1.0, 1.0]
    m.close()
    # chunked aggregation keeps today's refusals for wide keys and raw utf8 members
    _raises(pab, NOT_IMPLEMENTED, lambda: pab.aggregate_chunked([rb.column("k1"), rb.column("k2")], rb.column("v"), ["sum"], 4096),
            match="composite key needs 130 bits; only keys that pack into 64 bits")
    from pandasarrow_b200 import _lib
    from pandasarrow_b200._lib import PA_AGG
    from pandasarrow_b200.groupby import _CArg, _check, _options, _pack_args
    args, devs, schemas = _pack_args([pa.array([1, 2, 1], pa.int32()), pa.array(["a", "b", "a"])])
    va = _CArg(pa.array([1.0, 2.0, 3.0]))
    h = C.c_void_p()
    opt = _options(0)
    try:
        _raises(pab, NOT_IMPLEMENTED, lambda: _check(_lib.load().pa_groupby_aggregate_chunked_keys(
            devs, schemas, 2, C.byref(va.dev), C.byref(va.schema), PA_AGG["sum"], 2, C.byref(opt), C.byref(h))),
            match="utf8 keys inside a composite key: dictionary-encode that column")
    finally:
        for a in args:
            a.close()
        va.close()
    # the harness still encodes utf8 members for chunked aggregation
    mc = pab.aggregate_chunked([pa.array([1, 2, 1], pa.int32()), pa.array(["a", "b", "a"])], pa.array([1.0, 2.0, 3.0]), ["sum"], 2)
    assert mc.fetch("sum").to_pylist() == [4.0, 2.0]
    mc.close(); gb.close(); packed.close()


def test_twenty_million_rows_a_million_groups():
    import torch
    import pandasarrow_b200 as pab
    n, G = 20_000_000, 1_000_000
    gen = torch.Generator(device="cuda").manual_seed(7)
    ids = torch.randint(0, G, (n,), device="cuda", generator=gen)
    k1 = ids * 1_000_003 - 2**62
    k2 = (ids ^ 0x5555) * 0x7FFFFFFFFFFFFFC5 + (1 << 40)          # an odd multiplier: one value per id (int64 wraps)
    w = torch.randint(-10**9, 10**9, (n,), device="cuda", generator=gen)
    gb = pab.GroupBy(["k1", "k2"], {"k1": pab.DeviceColumn.from_torch(k1), "k2": pab.DeviceColumn.from_torch(k2)})
    r = gb.aggregate(pab.DeviceColumn.from_torch(w), ["count", "min", "max", "sum"])
    hid, hw = ids.cpu().numpy(), w.cpu().numpy()
    uniq, first, inv = np.unique(hid, return_index=True, return_inverse=True)
    order = np.argsort(first)                                   # groups in first-appearance order
    rank = np.empty_like(order)
    rank[order] = np.arange(len(order))
    gid = rank[inv]
    srt = np.argsort(gid, kind="stable")
    starts = np.flatnonzero(np.r_[True, np.diff(gid[srt]) != 0])
    ws = hw[srt]
    assert gb.groupSize() == len(uniq)
    assert np.array_equal(r["count"].to_numpy(), np.diff(np.r_[starts, n]))
    assert np.array_equal(r["min"].to_numpy(), np.minimum.reduceat(ws, starts))
    assert np.array_equal(r["max"].to_numpy(), np.maximum.reduceat(ws, starts))
    assert np.array_equal(r["sum"].to_numpy(), np.add.reduceat(ws, starts))
    assert np.array_equal(gb.unique(0).to_numpy(), k1.cpu().numpy()[first[order]])
    assert gb.key_hash_seed() == 0
    gb.close()
