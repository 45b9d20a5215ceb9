"""Sum-only dense passes (csrc/lowcard_known.cuh): once a full dense pass of the narrow set has been read back, later
passes on the handle report mode "dense-known" and give the bits of the full pass (and of PA_LC_NO_KNOWN=1, which
forces the full pass), against the oracle.  Needs a GPU: -m gpu."""

import numpy as np
import pyarrow as pa
import pytest

pytestmark = pytest.mark.gpu

FP_AGGS = ["sum", "mean", "count", "first"]
INT_AGGS = ["sum", "count", "first"]
SENTINEL = np.uint64(0x9E3779B97F4A7C15).astype(np.int64)   # common.cuh kEmptyKey: a regular key on this path


@pytest.fixture(scope="module")
def pab():
    import pandasarrow_b200 as p
    return p


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


def bits(res):
    """Every output as (null mask, raw 64-bit words): equality is bit for bit."""
    out = {}
    for a, arr in res.items():
        nulls = np.asarray(arr.is_null().to_numpy(zero_copy_only=False))
        v = np.asarray(arr.fill_null(0).to_numpy(zero_copy_only=False))
        out[a] = (nulls.tolist(), v.astype(v.dtype.newbyteorder("=")).view(np.uint8).tobytes())
    return out


def mode(gb):
    return gb.timing()["mode"]


def check_oracle(orc, rb, uniq, res, aggs):
    ora = orc.OracleGroupBy(rb, "k")
    want_keys = ora.unique().to_pylist()
    pos = {k: i for i, k in enumerate(uniq.to_pylist())}
    assert set(pos) == set(want_keys)
    p = np.array([pos[k] for k in want_keys])
    for a in aggs:
        want = np.asarray(ora.agg(a, "v", nthreads=4).to_numpy(zero_copy_only=False))
        got = np.asarray(res[a].to_numpy(zero_copy_only=False))[p]
        if a in ("sum", "mean") and got.dtype.kind == "f":
            np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-6, err_msg=a)
        else:
            assert np.array_equal(got, want, equal_nan=got.dtype.kind == "f"), a


def known_chain(pab, orc, monkeypatch, rb, keys, vals, aggs):
    """First pass full, two sum-only passes, one forced full pass: all bit-identical, and right."""
    gb = pab.GroupBy("k", {"k": keys, "v": vals})
    runs, modes = [], []
    for force_full in (False, False, False, True):
        if force_full:
            monkeypatch.setenv("PA_LC_NO_KNOWN", "1")
        runs.append(bits(gb.aggregate(vals, aggs)))
        modes.append(mode(gb))
        monkeypatch.delenv("PA_LC_NO_KNOWN", raising=False)
    assert modes == ["dense", "dense-known", "dense-known", "dense"]
    for r in runs[1:]:
        assert r == runs[0]
    res = gb.aggregate(vals, aggs)
    assert mode(gb) == "dense-known" and bits(res) == runs[0]
    check_oracle(orc, rb, gb.unique(), res, aggs)
    gb.close()


def dense_keys(rng, n, groups, base=0):
    return (base + rng.permutation(groups)[rng.integers(0, groups, n)]).astype(np.int64)


@pytest.mark.parametrize("groups", [1000, 256, 16, 2])
def test_known_pass_fp64(pab, orc, monkeypatch, groups):
    rng = np.random.default_rng(groups)
    n = (1 << 21) + 77                                  # a partial last row group as well
    k = dense_keys(rng, n, groups, base=-500)
    v = rng.normal(size=n) * 1e3
    rb = pa.record_batch({"k": pa.array(k), "v": pa.array(v)})
    known_chain(pab, orc, monkeypatch, rb, rb.column("k"), rb.column("v"), FP_AGGS)


def test_known_pass_fp64_specials(pab, orc, monkeypatch):
    rng = np.random.default_rng(7)
    n = 1 << 20
    k = dense_keys(rng, n, 600)
    v = rng.normal(size=n)
    v[k == 3] = -0.0                                    # a group of only negative zeros
    v[k == 5] = np.where(rng.random(int((k == 5).sum())) < 0.5, -0.0, 0.0)
    v[rng.random(n) < 1e-4] = np.nan
    v[(k == 7) & (rng.random(n) < 0.01)] = np.inf
    v[(k == 8) & (rng.random(n) < 0.01)] = -np.inf
    v[(k == 9) & (rng.random(n) < 0.01)] = np.inf
    v[(k == 9) & (rng.random(n) < 0.01)] = -np.inf
    rb = pa.record_batch({"k": pa.array(k), "v": pa.array(v)})
    known_chain(pab, orc, monkeypatch, rb, rb.column("k"), rb.column("v"), FP_AGGS)


@pytest.mark.parametrize("typ", [np.int64, np.uint64])
def test_known_pass_wrapping_integer_sums(pab, orc, monkeypatch, typ):
    rng = np.random.default_rng(11)
    n = (1 << 20) + 3
    k = dense_keys(rng, n, 100)
    info = np.iinfo(typ)
    v = rng.integers(info.max // 4, info.max, n, dtype=typ, endpoint=False)
    rb = pa.record_batch({"k": pa.array(k), "v": pa.array(v)})
    known_chain(pab, orc, monkeypatch, rb, rb.column("k"), rb.column("v"), INT_AGGS)


def test_known_pass_null_keys_and_sentinel(pab, orc, monkeypatch):
    rng = np.random.default_rng(13)
    n = 500_001
    k = dense_keys(rng, n, 300, base=int(SENTINEL) - 150)
    assert (k == SENTINEL).any()
    rb = pa.record_batch({"k": pa.array(k, mask=rng.random(n) < 0.02), "v": pa.array(rng.normal(size=n))})
    known_chain(pab, orc, monkeypatch, rb, rb.column("k"), rb.column("v"), FP_AGGS)


def test_known_pass_int32_keys_odd_slices(pab, orc, monkeypatch):
    rng = np.random.default_rng(17)
    n = 700_003
    k = pa.array(dense_keys(rng, n + 1, 900).astype(np.int32)).slice(1)
    v = pa.array(rng.normal(size=n + 1)).slice(1)
    rb = pa.record_batch({"k": k, "v": v})
    known_chain(pab, orc, monkeypatch, rb, k, v, FP_AGGS)


def test_nullable_values_between_clean_ones(pab, orc):
    rng = np.random.default_rng(19)
    n = 1 << 20
    k = pa.array(dense_keys(rng, n, 1000))
    clean = pa.array(rng.normal(size=n))
    holes = pa.array(rng.normal(size=n), mask=rng.random(n) < 0.1)
    gb = pab.GroupBy("k", {"k": k})
    first = bits(gb.aggregate(clean, FP_AGGS))
    assert mode(gb) == "dense"
    assert bits(gb.aggregate(clean, FP_AGGS)) == first and mode(gb) == "dense-known"
    res = gb.aggregate(holes, FP_AGGS)                  # counts differ from the group sizes: the full pass
    assert mode(gb) == "dense"
    check_oracle(orc, pa.record_batch({"k": k, "v": holes}), gb.unique(), res, FP_AGGS)
    assert bits(gb.aggregate(clean, FP_AGGS)) == first and mode(gb) == "dense-known"
    gb.close()


def test_keys_only_first_pass(pab, orc):
    rng = np.random.default_rng(23)
    n = 300_000
    k = pa.array(dense_keys(rng, n, 500))
    v = pa.array(rng.normal(size=n))
    gb = pab.GroupBy("k", {"k": k})
    uniq = gb.unique()                                  # groups found without a value column: no counts to keep
    r1 = gb.aggregate(v, FP_AGGS)
    assert mode(gb) == "dense"
    r2 = gb.aggregate(v, FP_AGGS)
    assert mode(gb) == "dense-known" and bits(r2) == bits(r1)
    assert gb.unique().equals(uniq)
    check_oracle(orc, pa.record_batch({"k": k, "v": v}), uniq, r2, FP_AGGS)
    gb.close()


def test_deferred_chains(pab, orc):
    import torch
    rng = np.random.default_rng(29)
    n = (1 << 22) + 5
    kn = dense_keys(rng, n, 1000)
    vn = rng.normal(size=n)
    keys = torch.from_numpy(kn).cuda()
    vals = torch.from_numpy(vn).cuda()
    dk, dv = pab.DeviceColumn.from_torch(keys), pab.DeviceColumn.from_torch(vals)
    ref = pab.GroupBy("k", {"k": dk})
    want = bits(ref.aggregate(dv, FP_AGGS))
    ref.close()
    gb = pab.GroupBy("k", {"k": dk})
    # the recording passes are superseded before anybody reads them: nothing is trusted until one is read back
    for _ in range(3):
        gb.aggregate(dv, FP_AGGS, fetch=False, wait=False)
    assert mode(gb) == "dense"
    assert bits({a: gb.fetch(a) for a in FP_AGGS}) == want
    for _ in range(3):
        gb.aggregate(dv, FP_AGGS, fetch=False, wait=False)
    assert mode(gb) == "dense-known"
    got = {a: gb.fetch(a) for a in FP_AGGS}
    assert bits(got) == want and gb.groupSize() == 1000
    check_oracle(orc, pa.record_batch({"k": pa.array(kn), "v": pa.array(vn)}), gb.unique(), got, FP_AGGS)
    # a key outside the recorded window (the caller rewrote the key column): the deferred sum-only pass aborts and
    # the full pass redoes it
    keys[12345] = 5000
    kn[12345] = 5000
    gb.aggregate(dv, FP_AGGS, fetch=False, wait=False)
    with pytest.raises(pab.PaError, match="group count changed"):
        gb.sync()
    gb.close()


def test_set_key_layout_drops_the_facts(pab):
    rng = np.random.default_rng(31)
    n = 400_000
    # a dictionary column packs into 6 bits below a constant int32 column: the key word is the dictionary index, dense
    a = pa.DictionaryArray.from_arrays(pa.array(rng.integers(0, 40, n).astype(np.int32)),
                                       pa.array(np.arange(40, dtype=np.int64) * 1000))
    b = pa.array(np.zeros(n, dtype=np.int32))
    v = pa.array(rng.normal(size=n))
    gb = pab.GroupBy(["a", "b"], {"a": a, "b": b})
    r1 = bits(gb.aggregate(v, FP_AGGS))
    assert mode(gb) == "dense"
    assert bits(gb.aggregate(v, FP_AGGS)) == r1 and mode(gb) == "dense-known"
    layout = gb.key_layout()
    layout.nullable[1] = 1                              # a null bit for column 1: the key words are packed anew
    gb.set_key_layout(layout)
    assert bits(gb.aggregate(v, FP_AGGS)) == r1 and mode(gb) == "dense"
    assert bits(gb.aggregate(v, FP_AGGS)) == r1 and mode(gb) == "dense-known"
    gb.close()


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


def test_sharded_step_with_row_base(pab, orc, single_rank_comm):
    rng = np.random.default_rng(37)
    n = 600_000
    k = pa.array(dense_keys(rng, n, 1000))
    v = pa.array(rng.normal(size=n))
    gb = pab.GroupBy("k", {"k": k}, row_base=123_456)
    steps, modes = [], []
    for _ in range(3):
        m = single_rank_comm.sharded_aggregate(gb, v, FP_AGGS)
        modes.append(mode(gb))
        steps.append(bits({a: m.fetch(a) for a in FP_AGGS}))
        if len(steps) == 3:
            uniq = m.unique()
            res = {a: m.fetch(a) for a in FP_AGGS}
        m.close()
    assert modes == ["dense", "dense-known", "dense-known"]
    assert steps[1] == steps[0] and steps[2] == steps[0]
    check_oracle(orc, pa.record_batch({"k": k, "v": v}), uniq, res, FP_AGGS)
    gb.close()
