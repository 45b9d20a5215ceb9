"""Composite keys across shards, on CPU: the key-layout agreement over gloo (world 2) and a numpy model of the packing
that shows why it is needed — a group packed under each shard's own layout can land on different owners, packed under
the agreed layout it lands on one.  The layouts are built by hand here; on a GPU they come from GroupBy.key_layout()."""
import ctypes as C
import os

import numpy as np
import pytest

from pandasarrow_b200 import distributed as D
from pandasarrow_b200._lib import PaKeyLayout


def layout(widths, bits, nullable, fps=None):
    l = PaKeyLayout()
    l.n_keys = len(widths)
    for j in range(len(widths)):
        l.width[j], l.bits[j], l.nullable[j] = widths[j], bits[j], nullable[j]
        l.dict_fingerprint[j] = 0 if fps is None else fps[j]
    return l


def pack_model(cols, nulls, lay):
    """Host twin of k_pack_keys (csrc/emit.cuh) with the shifts of layout_fields (csrc/capi.cu): column j takes
    bits[j] value bits and, when nullable[j], one null bit, in column order from bit 0."""
    out = np.zeros(len(cols[0]), dtype=np.uint64)
    shift = 0
    for j in range(lay.n_keys):
        raw = np.asarray(cols[j]).astype(np.int64).view(np.uint64)
        if lay.width[j] == 4:
            raw = raw & np.uint64(0xFFFFFFFF)
        b = lay.bits[j]
        v = raw & np.uint64((1 << b) - 1 if b < 64 else (1 << 64) - 1)
        if lay.nullable[j]:
            v = np.where(np.asarray(nulls[j], dtype=bool), np.uint64(1 << b), v)
        with np.errstate(over="ignore"):
            out |= v << np.uint64(shift)
        shift += b + lay.nullable[j]
    assert shift <= 64
    return out


def _worker(rank, world, path, q):
    import torch.distributed as dist
    os.environ.setdefault("GLOO_SOCKET_IFNAME", "lo")
    store = dist.FileStore(path, world)
    dist.init_process_group("gloo", store=store, rank=rank, world_size=world)
    out = {}

    class FakeGroupBy:                         # the layout of a shard, without a GPU
        def __init__(self, lay):
            self.lay, self.applied = lay, None

        def key_layout(self):
            return self.lay

        def set_key_layout(self, l):
            self.applied = l
    try:
        # int32 x dictionary(64): rank 0 has no null in k1, rank 1 none in k2
        g = FakeGroupBy(layout([4, 4], [32, 6], [0, 1] if rank == 0 else [1, 0], [0, 77]))
        a = D.agree_key_layout(g)
        out["agreed"] = (a.n_keys, list(a.width)[:2], list(a.bits)[:2], list(a.nullable)[:2], list(a.dict_fingerprint)[:2])
        out["applied"] = g.applied is not None and bytes(g.applied) == bytes(a)
        for what, lay in (("width", layout([4, 4], [32, 6], [0, 1], [0, 77]) if rank == 0 else layout([8, 4], [64, 6], [0, 1], [0, 77])),
                          ("dictionary", layout([4, 4], [32, 6], [0, 1], [0, 77 + rank])),
                          ("bits", layout([4, 4], [32, 6 + rank], [0, 1], [0, 77])),
                          ("64 bits", layout([4, 4], [32, 31], [rank, 1 - rank], [0, 0]))):
            g = FakeGroupBy(lay)
            try:
                D.agree_key_layout(g)
                out[what] = None
            except Exception as e:              # noqa: BLE001 — the message travels back to the test
                out[what] = (type(e).__name__, str(e), g.applied is None)
    finally:
        dist.destroy_process_group()
    q.put((rank, out))


def test_agree_key_layout_over_gloo(tmp_path):
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, str(tmp_path / "store"), q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for r in range(2):
        out = res[r]
        assert out["agreed"] == (2, [4, 4], [32, 6], [1, 1], [0, 77])       # nullable: OR over the ranks
        assert out["applied"]
        # every rank raises, and neither repacks
        for what, match in (("width", "widths differ"), ("dictionary", "one dictionary shared by all shards"),
                            ("bits", "value bits differ"), ("64 bits", "needs 65 bits")):
            name, msg, untouched = out[what]
            assert name == "PaError" and match in msg and untouched, (r, what, msg)


def test_agreed_layout_routes_a_group_to_one_owner():
    """Config 3 (int32 x dictionary<int32 -> utf8> of 64 symbols) sharded so that shard 0 has no null k1: under each
    shard's own layout the k2 field starts at bit 32 on shard 0 and at bit 33 on shard 1, so the same (k1, k2) packs to
    two words and, for most groups, two owners; under the agreed layout it is one word and one owner."""
    rng = np.random.default_rng(5)
    n, world = 20_000, 8
    k1 = rng.integers(0, 1000, n).astype(np.int32)
    k2 = rng.integers(0, 64, n).astype(np.int32)
    n1 = np.zeros(n, dtype=bool)
    n2 = rng.random(n) < 0.01
    own0 = layout([4, 4], [32, 6], [0, 1], [0, 9])
    own1 = layout([4, 4], [32, 6], [1, 1], [0, 9])
    agreed = D.agree_layouts([own0, own1])
    assert list(agreed.nullable)[:2] == [1, 1]
    w0, w1 = pack_model([k1, k2], [n1, n2], own0), pack_model([k1, k2], [n1, n2], own1)
    o0, o1 = D.owner_of(w0, world), D.owner_of(w1, world)
    assert (w0 != w1).mean() > 0.95 and (o0 != o1).mean() > 0.5
    wa = pack_model([k1, k2], [n1, n2], agreed)
    assert np.array_equal(wa, w1)                           # rank 1 already packs with it; rank 0 repacks
    # one word per group: the agreed words are a bijection of the (k1, k2-or-null) tuples
    tuples = set(zip(k1.tolist(), np.where(n2, -1, k2).tolist()))
    assert len(set(wa.tolist())) == len(tuples)


def test_full_width_key_packs_without_null_bits():
    """Two int32 columns without nulls use all 64 bits; negative values keep their 32-bit patterns."""
    k1 = np.array([-1, 0, 5, -2_147_483_648], dtype=np.int32)
    k2 = np.array([-1, 7, -5, 2_147_483_647], dtype=np.int32)
    lay = D.agree_layouts([layout([4, 4], [32, 32], [0, 0])] * 3)
    w = pack_model([k1, k2], [np.zeros(4, bool)] * 2, lay)
    assert w[0] == np.uint64((1 << 64) - 1)
    assert w[3] == np.uint64(0x7FFFFFFF_80000000)


def test_agree_rejects_malformed_layouts():
    from pandasarrow_b200 import PaError
    with pytest.raises(PaError, match="key columns"):
        D.agree_layouts([layout([4], [32], [0])])
    with pytest.raises(PaError, match="not a packable field"):
        D.agree_layouts([layout([4, 4], [33, 6], [0, 0])])
    with pytest.raises(PaError, match="number of key columns"):
        D.agree_layouts([layout([4, 4], [32, 6], [0, 0]), layout([4, 4, 4], [8, 8, 8], [0, 0, 0])])
    assert C.sizeof(PaKeyLayout) == 4 + 3 * 4 * 4 + 4 + 4 * 8
