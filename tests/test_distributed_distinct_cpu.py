"""Distinct-pair records (count_distinct across row-range shards) on CPU: world_size-2 gloo processes exchange
PA_DISTINCT_PAIR_WORDS-word records exactly as the NCCL ranks do, and a numpy model of the exchange — every shard's
distinct (key, value bits) set routed by owner_of, the owner's union counted per key — reproduces count_distinct on the
whole data.  No GPU needed."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

PW = 3


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _fake_pairs(rank, world, n):
    """Pair records this rank would send, grouped by owner: (key, value bits, flags); the bits word encodes the rank."""
    from pandasarrow_b200 import distributed as D
    rng = np.random.default_rng(300 + rank)
    keys = rng.integers(-300, 300, n).astype(np.int64)
    bits = (rng.integers(0, 1 << 40, n) << 8 | rank).astype(np.int64)
    flags = (keys % 17 == 0).astype(np.int64)                  # some pairs of the null key
    own = D.owner_of(keys, world, is_null=flags.astype(bool))
    order = np.argsort(own, kind="stable")
    rec = np.stack([keys, bits, flags], axis=1)[order]
    counts = [int((own == o).sum()) for o in range(world)]
    return rec, counts


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from pandasarrow_b200 import distributed as D
    from pandasarrow_b200._lib import PA_DISTINCT_PAIR_WORDS
    rec, counts = _fake_pairs(rank, world, 500)
    recv, rc = D.exchange_records(torch.from_numpy(rec), counts, words=PA_DISTINCT_PAIR_WORDS)
    recv = recv.numpy()
    ok = recv.shape[1] == PW and sum(rc) == len(recv)
    ok &= bool((D.owner_of(recv[:, 0], world, is_null=recv[:, 2].astype(bool)) == rank).all())
    off = 0
    for s in range(world):   # grouped by source rank, every word intact
        seg = recv[off:off + rc[s]]
        exp_rec, exp_counts = _fake_pairs(s, world, 500)
        e_off = sum(exp_counts[:rank])
        ok &= np.array_equal(seg, exp_rec[e_off:e_off + exp_counts[rank]])
        off += rc[s]
    q.put((rank, bool(ok)))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(120)
def test_gloo_world2_exchange_of_distinct_pairs():
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=100) for _ in range(world)]
    for p in procs:
        p.join(timeout=30)
        assert p.exitcode == 0
    for rank, ok in results:
        assert ok, f"rank {rank}: 3-word pair records not delivered intact, grouped by source"


def _shard_pairs(keys, knull, vals, vnull):
    """What one shard keeps: its distinct (key, null-key flag, value bits) of the non-null values."""
    bits = vals.view(np.uint64)
    keep = ~vnull
    return set(zip(np.where(knull, 0, keys)[keep].tolist(), knull[keep].tolist(), bits[keep].tolist()))


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_owner_union_of_shard_pairs_is_count_distinct(world):
    from pandasarrow_b200 import distributed as D
    rng = np.random.default_rng(world)
    n = 20_000
    keys = rng.integers(0, 200, n).astype(np.int64)
    knull = rng.random(n) < 0.03
    vals = rng.integers(-6, 6, n).astype(np.float64) / 2
    vals[rng.random(n) < 0.05] = -0.0
    nan = np.float64(np.nan).view(np.uint64)
    payloads = np.array([nan, nan | np.uint64(1), nan | np.uint64(1 << 63)], np.uint64).view(np.float64)
    is_nan = rng.random(n) < 0.05
    vals[is_nan] = payloads[rng.integers(0, 3, is_nan.sum())]
    vals[rng.random(n) < 0.01] = np.inf
    vnull = rng.random(n) < 0.1
    # whole data: distinct non-null bit patterns per group (the null key is one group)
    want = {}
    for k, kn, b, vn in zip(keys.tolist(), knull.tolist(), vals.view(np.uint64).tolist(), vnull.tolist()):
        g = None if kn else k
        want.setdefault(g, set())
        if not vn:
            want[g].add(b)
    want = {g: len(s) for g, s in want.items()}
    # shards -> routed pairs -> per-owner union
    bounds = [D.shard_rows(n, world, r) for r in range(world)]
    inbox = [set() for _ in range(world)]
    sent = 0
    for b, e in bounds:
        pairs = _shard_pairs(keys[b:e], knull[b:e], vals[b:e], vnull[b:e])
        sent += len(pairs)
        for k, kn, bits in pairs:
            o = int(D.owner_of(np.array([k], np.int64), world, is_null=np.array([kn]))[0])
            inbox[o].add((k, kn, bits))
    assert sent >= sum(len(s) for s in inbox)
    got = {}
    for o, s in enumerate(inbox):
        for k, kn, _ in s:
            g = None if kn else k
            if kn:
                assert o == 0                                   # the null key lives on rank 0
            got[g] = got.get(g, 0) + 1
    assert {g: c for g, c in want.items() if c} == got
    assert want[None] > 0 and len({b for b in vals.view(np.uint64)[np.isnan(vals) & ~vnull].tolist()}) == 3
