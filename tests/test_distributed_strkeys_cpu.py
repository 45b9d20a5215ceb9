"""utf8 keys across shards, on CPU: world-size-2 gloo runs of the hash-seed agreement and of the key length / byte
exchange, and a numpy model of the layout the export writes (per owner, the key bytes in record order) and of the
owner's representative rule (the record with the smallest global first row), checked against Python string grouping."""
import os
import socket

import numpy as np
import pytest


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _run(fn, world=2):
    import torch.multiprocessing as mp
    port = _free_port()
    mp.spawn(_entry, args=(fn, world, port), nprocs=world, join=True)


def _entry(rank, fn, world, port):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        fn(rank, world)
    finally:
        dist.destroy_process_group()


class _FakeHandle:
    """What agree_key_hash_seed needs of a GroupBy: its seed, and a setter."""

    def __init__(self, seed):
        self.seed, self.set_calls = seed, []

    def key_hash_seed(self):
        return self.seed

    def set_key_hash_seed(self, seed):
        self.set_calls.append(seed)
        self.seed = seed


def _seed_worker(rank, world):
    from pandasarrow_b200 import distributed as D
    from pandasarrow_b200.groupby import PaError
    g = _FakeHandle(0)
    assert D.agree_key_hash_seed(g) == (0, True) and g.seed == 0
    g = _FakeHandle(rank)                    # rank 1's own check moved its seed
    assert D.agree_key_hash_seed(g) == (1, False) and g.seed == 1
    assert D.agree_key_hash_seed(g) == (1, True)
    g = _FakeHandle(4 if rank else 2)
    with pytest.raises(PaError, match="four differently seeded"):
        D.agree_key_hash_seed(g)


def test_agree_key_hash_seed_gloo():
    _run(_seed_worker)


def _strings(rank):
    return [["", "ü", "abc"], ["日本語", "x" * 70]][rank]


def _exchange_worker(rank, world):
    import torch
    from pandasarrow_b200 import distributed as D
    # rank r sends to rank p: the strings _strings(r)[p:] ... as records (lengths) + bytes
    mine = _strings(rank)
    per_owner = [mine[:1], mine[1:]]
    lens = torch.tensor([len(s.encode()) for o in per_owner for s in o], dtype=torch.int32)
    data = torch.tensor(list(b"".join(s.encode() for o in per_owner for s in o)), dtype=torch.uint8)
    counts = [len(o) for o in per_owner]
    nbytes = [sum(len(s.encode()) for s in o) for o in per_owner]
    rlen, rdata, rc, rb = D.exchange_key_strings(lens, data, counts, nbytes)
    want = [_strings(s)[:1] if rank == 0 else _strings(s)[1:] for s in range(world)]
    assert rc == [len(w) for w in want] and rb == [sum(len(x.encode()) for x in w) for w in want]
    flat = [x for w in want for x in w]
    assert rlen.tolist() == [len(x.encode()) for x in flat]
    off = np.concatenate([[0], np.cumsum(rlen.numpy())])
    assert [bytes(rdata[off[i]:off[i + 1]].tolist()).decode() for i in range(len(flat))] == flat


def test_exchange_key_strings_gloo():
    _run(_exchange_worker)


def export_model(keys, row_base, world):
    """The export of one shard: groups in first-appearance order (the local first row), routed by owner, written owner
    after owner; within an owner the records are in any order (here: a shuffled one, as the scatter's atomics leave them),
    and the key bytes follow the records as written.  Returns (records [(owner, global first row, key)], lengths, bytes)."""
    rng = np.random.default_rng(row_base + 1)
    first = {}
    for i, k in enumerate(keys):
        first.setdefault(k, i)
    groups = list(first.items())
    owner = {k: (0 if k is None else hash_owner(k, world)) for k, _ in groups}
    recs = []
    for o in range(world):
        seg = [(o, row_base + r, k) for k, r in groups if owner[k] == o]
        recs += [seg[j] for j in rng.permutation(len(seg))]
    lengths = [0 if k is None else len(k.encode()) for _, _, k in recs]
    data = b"".join(b"" if k is None else k.encode() for _, _, k in recs)
    return recs, lengths, data


def hash_owner(s, world):
    import zlib
    return zlib.crc32(s.encode()) % world


def test_export_layout_and_representative_model():
    """Owner side of the model: read every record's bytes back from the pool by the scanned lengths, group by key bytes,
    and take as representative the record with the smallest global first row: the groups and their first rows are what
    Python string grouping over the whole column gives, and each group's bytes are its first string."""
    rng = np.random.default_rng(5)
    world, n = 3, 3000
    pool = ["", "é", "ab", "日本", "x" * 33] + [f"k{i}" for i in range(40)]
    col = [None if rng.random() < 0.03 else pool[j] for j in rng.integers(0, len(pool), n)]
    bounds = [(0, 1000), (1000, 1000), (1000, 3000)]            # shard 1 is empty
    exports = [export_model(col[b:e], b, world) for b, e in bounds]
    merged = {}
    for o in range(world):
        recs, lens, chunks = [], [], []
        for recs_s, lens_s, data_s in exports:
            off = np.concatenate([[0], np.cumsum(lens_s)]).astype(np.int64)
            for i, (ow, fr, k) in enumerate(recs_s):
                if ow == o:
                    recs.append((fr, k)); lens.append(lens_s[i]); chunks.append(data_s[off[i]:off[i + 1]])
        reps = {}
        for (fr, k), b in zip(recs, chunks):
            key = None if k is None else b.decode()
            assert key == k, "bytes follow their record"
            if key not in reps or fr < reps[key]:
                reps[key] = fr
        for k, fr in reps.items():
            assert k not in merged, "a key has one owner"
            merged[k] = fr
    first = {}
    for i, k in enumerate(col):
        first.setdefault(k, i)
    assert merged == first
    assert [k for k, _ in sorted(merged.items(), key=lambda t: t[1])] == list(first)
