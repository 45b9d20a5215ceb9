"""Stage-2 records (product / variance / stddev across row-range shards) on CPU: world_size-2 gloo processes exchange
PA_PARTIAL_WORDS_STAGE2-word records exactly as the NCCL ranks do, and a numpy model of the owner-side merge — per-shard
two-pass terms combined with Chan's update and a product in source-rank order (k_merge_fold<true>, csrc/merge.cuh) —
is checked against the two-pass formula on the whole group.  No GPU needed."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

W = 13


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _fake_records(rank, world, n):
    """Stage-2 records this rank would send: key k is owned by owner_of(k); every word encodes (rank, key, word)."""
    from pandasarrow_b200 import distributed as D
    rng = np.random.default_rng(200 + rank)
    keys = np.unique(rng.integers(0, 500, n).astype(np.int64))   # one record per key and source, like real partials
    own = D.owner_of(keys, world)
    order = np.argsort(own, kind="stable")
    keys, own = keys[order], own[order]
    rec = (keys[:, None] * 1000 + rank * 100 + np.arange(W)[None, :]).astype(np.int64)
    rec[:, 0] = keys
    counts = [int((own == o).sum()) for o in range(world)]
    return rec, counts


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from pandasarrow_b200 import distributed as D
    from pandasarrow_b200._lib import PA_PARTIAL_WORDS_STAGE2
    rec, counts = _fake_records(rank, world, 300)
    recv, rc = D.exchange_records(torch.from_numpy(rec), counts, words=PA_PARTIAL_WORDS_STAGE2)
    recv = recv.numpy()
    ok = recv.shape[1] == W and sum(rc) == len(recv)
    ok &= bool((D.owner_of(recv[:, 0], world) == rank).all())
    off = 0
    for s in range(world):   # grouped by source rank, every word intact
        seg = recv[off:off + rc[s]]
        exp_rec, exp_counts = _fake_records(s, world, 300)
        e_off = sum(exp_counts[:rank])
        ok &= np.array_equal(seg, exp_rec[e_off:e_off + exp_counts[rank]])
        off += rc[s]
    q.put((rank, bool(ok)))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(120)
def test_gloo_world2_exchange_of_stage2_records():
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
        assert ok, f"rank {rank}: 13-word records not delivered intact, grouped by source"


def _shard_terms(x):
    """What one shard ships: count, the mean the second pass used (sum / count), M2 around it, the product."""
    n = len(x)
    if n == 0:
        return 0, 0.0, 0.0, 1.0
    mean = x.sum() / n
    with np.errstate(invalid="ignore"):          # inf - inf: NaN, as on the device
        return n, mean, float(((x - mean) ** 2).sum()), float(np.prod(x))


def _merge(terms):
    """k_merge_fold<true>: sources in rank order, empty ones skipped, Chan's update of (n, mean, M2), product."""
    n, mean, m2, prod = 0, 0.0, 0.0, 1.0
    for nb, mb, m2b, pb in terms:
        if nb == 0:
            continue
        prod *= pb
        if n == 0:
            n, mean, m2 = nb, mb, m2b
            continue
        n2 = n + nb
        d = mb - mean
        m2 += m2b + d * d * n * nb / n2
        mean += d * nb / n2
        n = n2
    return n, m2, prod


def test_chan_merge_model_matches_two_pass():
    rng = np.random.default_rng(2024)
    worst = 0.0
    for trial in range(2000):
        shards = int(rng.integers(2, 9))
        size = int(rng.integers(1, 400))
        x = rng.normal(rng.uniform(-5, 5), rng.uniform(0.01, 10), size)
        if trial % 3 == 0:   # shards of one group whose means lie +-1e6 apart
            x += np.where(rng.random(size) < 0.5, 1e6, -1e6)
        cuts = np.sort(rng.integers(0, size + 1, shards - 1))
        parts = np.split(x, cuts)                       # row-range shards, some of them empty
        n, m2, _ = _merge([_shard_terms(p) for p in parts])
        assert n == size
        var = m2 / n
        want = np.mean((x - x.mean()) ** 2)
        worst = max(worst, abs(var - want) / max(want, np.mean(x * x)))
    assert worst <= 1e-12, worst


def test_chan_merge_model_edges_and_products():
    nan, inf = float("nan"), float("inf")
    # a constant group split over shards: exactly 0
    assert _merge([_shard_terms(np.full(k, 2.5)) for k in (3, 0, 2, 5)])[1] == 0.0
    # NaN or inf in one shard: NaN; the product carries the inf
    n, m2, prod = _merge([_shard_terms(np.array([1.0, 2.0])), _shard_terms(np.array([nan]))])
    assert np.isnan(m2) and np.isnan(prod)
    n, m2, prod = _merge([_shard_terms(np.array([2.0])), _shard_terms(np.array([inf, 1.0]))])
    assert np.isnan(m2) and prod == inf
    # float products in rank order against the product of the whole group
    rng = np.random.default_rng(5)
    for _ in range(200):
        x = np.where(rng.random(300) < 0.3, -1.0, 1.0) * np.exp(rng.normal(0, 0.05, 300))
        parts = np.split(x, np.sort(rng.integers(0, 301, 4)))
        got = _merge([_shard_terms(p) for p in parts])[2]
        want = float(np.prod(x))
        assert abs(got - want) <= 1e-12 * abs(want)
    # integer products wrap: the rank-order product of the shards' wrapped products is the wrapped whole product
    v = np.array([3] * 70 + [-7, 11, 13], dtype=np.int64)
    with np.errstate(over="ignore"):
        whole = np.prod(v.astype(np.uint64), dtype=np.uint64)
        parts = [np.prod(p.astype(np.uint64), dtype=np.uint64) for p in np.split(v, [30, 50, 71])]
        merged = np.uint64(1)
        for p in parts:
            merged = merged * p
    assert merged == whole
