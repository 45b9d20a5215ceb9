"""Multi-GPU group-by: one process per GPU, rows sharded by contiguous range (SURVEY.md §8e).

    local aggregate (stages 1-3 on this rank's shard)
      -> partial records bucketed by owner = hash(key) % world   (CUDA, pa_groupby_partials_*)
      -> all-to-all of counts, then of records                   (torch.distributed: NCCL over NVLink)
      -> merge by key in source-rank order + order by global first row   (CUDA, pa_merge_create)

Product / variance / stddev take the counted exchange with PA_PARTIAL_WORDS_STAGE2-word records, which also carry every
shard's two-pass terms (M2 and product); the merge combines them in source-rank order.  All / any take the counted
exchange too (min / max of the 0 / 1 values).  Count_distinct needs a second exchange: every shard's distinct
(key, value) pairs, PA_DISTINCT_PAIR_WORDS words each, go to the key's owner, which counts them without duplicates.

Each rank ends up owning the groups with hash(key) % world == rank; `gather_result` concatenates
the owners' results on every rank and restores global first-appearance order.

Composite keys (group_by(["k1", "k2"])) travel as their packed 64-bit word.  How a shard packs depends on its data: a
column carries a null bit only when the shard's slice of it has nulls, and a dictionary column is packed as its codes.
So before the local pass every shard agrees on one layout (agree_key_layout: the null bits of all shards, identical
widths and dictionaries) and repacks to it; then the same group is the same word, and has the same owner, everywhere.
A utf8 column in a sharded composite key must therefore be dictionary-encoded ONCE, over the whole column, before it
is sliced into shards: per-shard `dictionary_encode()` gives every shard its own codes, and the agreement fails with a
dictionary-fingerprint error instead of merging different strings into one group.

A single utf8 / large_utf8 key (group_by("name")) is grouped by a seeded 64-bit hash of its bytes, and its records carry
that hash.  Every record therefore travels with its group's key bytes (partials_export_utf8, exchange_key_strings),
and the owner compares the bytes of every record of a merged group with its representative's (merge_key_strings).
All shards must hash with one seed: a shard whose own byte check found a collision has moved to the next seed, so
before the exchange the shards agree on the largest (agree_key_hash_seed) and re-aggregate when it is not theirs.  A
collision that only the owner sees (two strings of different shards, one hash) makes every rank retry with the next
seed; four seeds at most, as on one GPU.

torch.distributed is plumbing only (rendezvous + the collective); the exchange helpers work on any
backend, which is what the world_size-2 gloo tests exercise on CPU.
"""
from __future__ import annotations

import functools
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from ._lib import PA_AGG, PA_AGG_STAGE2, PA_DISTINCT_PAIR_WORDS, PA_PARTIAL_WORDS, PA_PARTIAL_WORDS_STAGE2

REC_KEY, REC_FLAGS, REC_SUM, REC_DSUM, REC_COUNT, REC_FIRST_ROW = 0, 1, 2, 3, 4, 5


def shard_rows(n_total: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous row range [begin, end) of `rank` (rank r owns rows [r*N/P, (r+1)*N/P))."""
    return (rank * n_total) // world, ((rank + 1) * n_total) // world


def _mix64(k: np.ndarray) -> np.ndarray:
    """Host twin of hash_key64 (csrc/common.cuh)."""
    k = k.astype(np.uint64, copy=True)
    with np.errstate(over="ignore"):
        k ^= k >> np.uint64(33)
        k *= np.uint64(0xFF51AFD7ED558CCD)
        k ^= k >> np.uint64(33)
        k *= np.uint64(0xC4CEB9FE1A85EC53)
        k ^= k >> np.uint64(33)
    return k


def owner_of(keys: np.ndarray, world: int, is_null: Optional[np.ndarray] = None) -> np.ndarray:
    """Owner rank of every key (null keys live on rank 0) — must match owner_of() in csrc/merge.cuh."""
    o = (_mix64(np.asarray(keys).view(np.uint64) if np.asarray(keys).dtype.itemsize == 8 else np.asarray(keys)) %
         np.uint64(world)).astype(np.int64)
    if is_null is not None:
        o[np.asarray(is_null, dtype=bool)] = 0
    return o


def exchange_records(send, send_counts: Sequence[int], group=None, words: int = PA_PARTIAL_WORDS):
    """All-to-all of fixed-size records.  `send`: int64 tensor [sum(send_counts), words] (PA_PARTIAL_WORDS,
    PA_PARTIAL_WORDS_STAGE2 for stage-2 records, PA_DISTINCT_PAIR_WORDS for distinct pairs), grouped by destination rank.  Returns (recv tensor grouped by source
    rank, recv_counts)."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    assert len(send_counts) == world
    dev = send.device
    sc = torch.tensor(list(send_counts), dtype=torch.int64, device=dev)
    rc = torch.empty(world, dtype=torch.int64, device=dev)
    dist.all_to_all_single(rc, sc, group=group)
    recv_counts = [int(x) for x in rc.tolist()]
    recv = torch.empty((sum(recv_counts), words), dtype=torch.int64, device=dev)
    w = words
    dist.all_to_all_single(recv.view(-1), send.reshape(-1), output_split_sizes=[c * w for c in recv_counts],
                           input_split_sizes=[int(c) * w for c in send_counts], group=group)
    return recv, recv_counts


def exchange_key_strings(lengths, data, send_counts: Sequence[int], send_bytes: Sequence[int], group=None):
    """All-to-all of a utf8 key's strings next to exchange_records: `lengths` (int32, one per record, grouped by
    destination like the records, send_counts of them per rank) and `data` (uint8, send_bytes[p] bytes for rank p).
    Returns (recv lengths, recv bytes, recv record counts, recv byte counts), grouped by source rank."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    assert len(send_counts) == world and len(send_bytes) == world
    dev = lengths.device
    sc = torch.tensor([[int(c), int(b)] for c, b in zip(send_counts, send_bytes)], dtype=torch.int64, device=dev)
    rc = torch.empty_like(sc)
    dist.all_to_all_single(rc.view(-1), sc.view(-1), group=group)
    recv_counts = [int(x) for x in rc[:, 0].tolist()]
    recv_bytes = [int(x) for x in rc[:, 1].tolist()]
    rlen = torch.empty(sum(recv_counts), dtype=lengths.dtype, device=dev)
    dist.all_to_all_single(rlen, lengths.reshape(-1), output_split_sizes=recv_counts, input_split_sizes=[int(c) for c in send_counts],
                           group=group)
    rdata = torch.empty(sum(recv_bytes), dtype=data.dtype, device=dev)
    dist.all_to_all_single(rdata, data.reshape(-1), output_split_sizes=recv_bytes, input_split_sizes=[int(b) for b in send_bytes],
                           group=group)
    return rlen, rdata, recv_counts, recv_bytes


def agree_key_hash_seed(gb, group=None) -> Tuple[int, bool]:
    """One hash seed for a utf8 key on every shard: all_reduce MAX of the seeds (any torch.distributed backend), set on
    `gb` (which drops its groups when the seed changes).  Returns (agreed seed, whether every shard already hashed with
    it); when not, every shard aggregates again.  PaError on every rank when the agreed seed is past the fourth."""
    import torch
    import torch.distributed as dist
    from .groupby import PaError
    mine = gb.key_hash_seed()
    t = torch.tensor([mine, -mine], dtype=torch.int64)       # (max, -min) in one reduction
    if dist.get_backend(group) == "nccl":
        t = t.cuda()
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    hi, lo = int(t[0]), -int(t[1])
    if hi >= MAX_HASH_SEEDS:
        raise PaError(4, "utf8 keys: four differently seeded 64-bit hashes all collided")
    gb.set_key_hash_seed(hi)
    return hi, lo == hi


MAX_HASH_SEEDS = 4   # as on one GPU (the library's utf8 key check)


def _utf8(gb) -> bool:
    return len(getattr(gb, "key_names", ())) == 1 and getattr(gb, "key_formats", [None])[0] in ("u", "U")


def agree_key_layout(gb, group=None):
    """All-gather the composite key layout of every shard's GroupBy (any torch.distributed backend), agree on one
    (pa_key_layout_agree: nullable wherever any shard has nulls; widths, bits and dictionaries must match, else PaError
    on every rank) and repack `gb` to it.  Returns the agreed PaKeyLayout."""
    import torch
    import torch.distributed as dist
    from ._lib import PaKeyLayout
    from .groupby import PaError
    world = dist.get_world_size(group)
    err = None
    try:
        mine = gb.key_layout()
    except PaError as e:          # still take part in the gather (n_keys = 0): every rank then fails together
        err, mine = e, PaKeyLayout()
    t = torch.tensor(list(bytes(mine)), dtype=torch.uint8)
    if dist.get_backend(group) == "nccl":
        t = t.cuda()
    parts = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(parts, t, group=group)
    if err is not None:
        raise err
    agreed = agree_layouts([PaKeyLayout.from_buffer_copy(bytes(p.cpu().tolist())) for p in parts])
    gb.set_key_layout(agreed)
    return agreed


def agree_layouts(layouts):
    """pa_key_layout_agree over every shard's PaKeyLayout: the one layout all of them pack with (PaError when they
    cannot agree)."""
    import ctypes as C
    from . import _lib
    from ._lib import PaKeyLayout
    from .groupby import _check
    all_ = (PaKeyLayout * len(layouts))(*layouts)
    agreed = PaKeyLayout()
    _check(_lib.load().pa_key_layout_agree(all_, len(layouts), C.byref(agreed)))
    return agreed


def _composite(gb) -> bool:
    return len(getattr(gb, "key_names", ())) > 1


class Comm:
    """pa_comm (include/pa_b200.h): an NCCL communicator owned by libpa_b200.so.  The unique id travels over the
    already initialised torch.distributed group (any backend); after that the whole sharded step — local pass, owner
    bucketing, count / record exchange, merge — is ONE C call (pa_groupby_sharded_aggregate), and this module is
    just its caller."""

    def __init__(self, group=None, device: Optional[int] = None):
        import ctypes as C
        import torch
        import torch.distributed as dist
        from . import _lib
        from .groupby import _check
        L = _lib.load()
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        dev = torch.cuda.current_device() if device is None else device
        buf = (C.c_uint8 * 128)()
        if rank == 0:
            _check(L.pa_comm_unique_id(buf, 128))
        t = torch.tensor(list(buf), dtype=torch.uint8)
        if dist.get_backend(group) == "nccl":
            t = t.cuda()
        dist.broadcast(t, src=0, group=group)
        raw = bytes(t.cpu().tolist())
        self._h = C.c_void_p()
        self.world, self.rank, self.device = world, rank, dev
        _check(L.pa_comm_create(raw, world, rank, dev, C.byref(self._h)))
        self._L = L

    def sharded_aggregate(self, gb, values, aggs: Sequence[str]):
        """One multi-GPU step; returns the owner-side MergedGroupBy."""
        import ctypes as C
        from ._lib import PA_AGG
        from .groupby import MergedGroupBy, _CArg, _check
        mask = 0
        for a in aggs:
            mask |= PA_AGG[a]
        arg = _CArg(values)
        h = C.c_void_p()
        try:
            _check(self._L.pa_groupby_sharded_aggregate(gb._h, self._h, C.byref(arg.dev), C.byref(arg.schema), mask, C.byref(h)))
        finally:
            arg.close()
        m = MergedGroupBy._from_handle(h)
        if _composite(gb):
            m._adopt_keys(gb.key_names, gb._dicts)
        return m

    def key_strings_info(self) -> Dict[str, int]:
        """utf8 key exchange of the last step (pa_comm_last_key_strings): key bytes sent and received, the agreed hash
        seed and the attempts the step took; zeros for a step without a utf8 key."""
        import ctypes as C
        from .groupby import _check
        sent, recv, seed, attempts = C.c_int64(), C.c_int64(), C.c_uint64(), C.c_int32()
        _check(self._L.pa_comm_last_key_strings(self._h, C.byref(sent), C.byref(recv), C.byref(seed), C.byref(attempts)))
        return {"bytes_sent": sent.value, "bytes_received": recv.value, "seed": seed.value, "attempts": attempts.value}

    def key_layout_info(self) -> Dict[str, float]:
        """Composite-key agreement of the last step (pa_comm_last_key_layout): device ms of the layout gather and of the
        repack (0 when none happened)."""
        import ctypes as C
        from .groupby import _check
        a, r = C.c_double(), C.c_double()
        _check(self._L.pa_comm_last_key_layout(self._h, C.byref(a), C.byref(r)))
        return {"agree_ms": a.value, "repack_ms": r.value}

    def phases(self) -> Dict[str, float]:
        import ctypes as C
        from .groupby import _check
        p = (C.c_double * 5)()
        _check(self._L.pa_comm_last_phases(self._h, p))
        return {"local_ms": p[0], "export_ms": p[1], "exchange_ms": p[2], "merge_ms": p[3], "total_ms": p[4]}

    def exchange_info(self) -> Dict[str, int]:
        """Record format of the last step (pa_comm_last_exchange)."""
        import ctypes as C
        from .groupby import _check
        rb, un, slots = C.c_int32(), C.c_int32(), C.c_int64()
        _check(self._L.pa_comm_last_exchange(self._h, C.byref(rb), C.byref(un), C.byref(slots)))
        return {"record_bytes": rb.value, "unordered_export": bool(un.value), "merge_table_slots": slots.value}

    def distinct_info(self) -> Dict[str, int]:
        """count_distinct exchange of the last step (pa_comm_last_distinct); zeros when it computed none."""
        import ctypes as C
        from .groupby import _check
        sent, recv, slots = C.c_int64(), C.c_int64(), C.c_int64()
        _check(self._L.pa_comm_last_distinct(self._h, C.byref(sent), C.byref(recv), C.byref(slots)))
        return {"pairs_sent": sent.value, "pairs_received": recv.value, "set_slots": slots.value}

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._L.pa_comm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


PADDED_BLOCK_RECORDS = 2048   # padded exchange: up to this many groups per rank (180 KB per peer block)


def exchange_padded(send_blocks, group=None):
    """Equal-split all-to-all of fixed-size blocks: send_blocks[p] goes to rank p, the result's block s came
    from rank s.  No counts are exchanged and nothing is read back: the whole step stays stream ordered."""
    import torch
    import torch.distributed as dist
    recv = torch.empty_like(send_blocks)
    dist.all_to_all_single(recv.view(-1), send_blocks.view(-1), group=group)
    return recv


def sharded_aggregate(gb, values, aggs: Sequence[str], value_format: str, key_format, group=None, stream=None,
                      padded: Optional[bool] = None, wait: bool = True, tail_stream=None):
    """Run the whole multi-GPU step for this rank.  `gb` is this rank's GroupBy over its row shard
    (created with row_base = first global row of the shard).  Returns the owner-side MergedGroupBy.

    Composite key: the shards first agree on one key layout (agree_key_layout, one all-gather); `key_format` may then
    be the list of key column formats, or None to take them (and the dictionaries unique() wraps) from `gb`.

    With few groups (<= PADDED_BLOCK_RECORDS on this rank) the partials travel in fixed-size blocks: one
    stream-ordered export kernel, one equal-split all-to-all, one merge — no host round trip in between.  A rank
    with more groups sends an overflow marker to every peer, so all ranks fall back to the counted exchange
    together.  `stream` must be the current torch stream for the padded path (it is in bench.py).

    wait=False (padded path only): nothing is read back at all — local pass, export, exchange and merge are just
    queued, so consecutive steps pipeline; the first call on the returned handle that needs a result completes
    it (and raises PaError if a rank had overflowed: rerun that step with wait=True).

    product / variance / stddev in `aggs`: always the counted exchange (the padded blocks hold PA_PARTIAL_WORDS-word
    records only), with stage-2 records.  all / any / count_distinct: the counted exchange as well; count_distinct then
    exchanges every shard's distinct pairs (exchange_records with words=PA_DISTINCT_PAIR_WORDS) and merges them into the
    owner's handle.

    tail_stream (a torch.cuda.Stream, padded path only): the exchange and the merge run on it, behind an event recorded
    after the export — the handle's own stream is free for the next step's local pass while this step's records travel
    and merge (the serial tail is launch / NCCL latency on a handful of CTAs).

    A single utf8 / large_utf8 key takes the counted exchange: the shards agree on a hash seed, the records travel with
    their key bytes, the owner checks and attaches the strings, and an all-reduce of the collision flag decides together
    whether every rank retries with the next seed.  `key_format` may be None (taken from `gb`)."""
    import torch
    import torch.distributed as dist
    from .groupby import MergedGroupBy, PaError
    world = dist.get_world_size(group)
    dev = torch.device("cuda", torch.cuda.current_device())
    stage2 = any(PA_AGG[a] & PA_AGG_STAGE2 for a in aggs)
    distinct = "count_distinct" in aggs
    if padded is None:
        padded = stream is not None and stream == torch.cuda.current_stream(dev).cuda_stream
    padded = padded and not stage2 and not any(a in ("all", "any", "count_distinct") for a in aggs)
    if _utf8(gb):
        return _sharded_utf8(gb, values, aggs, value_format, key_format or gb.key_formats[0], group, stream, dev, world)
    composite = _composite(gb)
    if composite:
        layout = agree_key_layout(gb, group)
        key_formats = list(key_format) if isinstance(key_format, (list, tuple)) else gb.key_formats
        key_format = "L"            # the records carry the packed word

    def adopt(merged):
        if composite:
            merged.set_composite_key(layout, key_formats, gb.key_names, gb._dicts)
        return merged
    # padded path: the local pass is only queued (no status read-back); export, exchange and merge are queued
    # behind it, so the host never waits before the merge's own result read.  A local pass that did not fit
    # the optimistic path makes the export send overflow markers, and everything is redone synchronously below.
    gb.aggregate(values, aggs, fetch=False, wait=not padded)
    if padded:
        cap = PADDED_BLOCK_RECORDS
        send = torch.empty((world, cap + 1, PA_PARTIAL_WORDS), dtype=torch.int64, device=dev)
        gb.partials_export_padded(world, send.data_ptr(), cap)
        try:
            if tail_stream is None:
                recv = exchange_padded(send, group)
                merged = adopt(MergedGroupBy(recv.data_ptr(), [0] * world, aggs, value_format, key_format, device=dev.index,
                                             stream=stream, padded_block_records=cap))
            else:
                done = torch.cuda.Event()
                done.record(torch.cuda.current_stream(dev))
                send.record_stream(tail_stream)
                with torch.cuda.stream(tail_stream):
                    tail_stream.wait_event(done)
                    recv = exchange_padded(send, group)
                    merged = adopt(MergedGroupBy(recv.data_ptr(), [0] * world, aggs, value_format, key_format, device=dev.index,
                                                 stream=tail_stream.cuda_stream, padded_block_records=cap))
            merged._keep = (send, recv)
            if wait:
                merged.groupSize()          # completes the merge; raises if any rank sent the overflow marker
            return merged
        except PaError as e:
            if "padded block" not in str(e):
                raise

    def counted_exchange(count, export, words):
        counts = count(world)
        send = torch.empty((max(sum(counts), 1), words), dtype=torch.int64, device=dev)
        export(world, send.data_ptr(), send.shape[0])
        recv, recv_counts = exchange_records(send[:sum(counts)], counts, group, words=words)
        torch.cuda.synchronize()
        return send, recv, recv_counts

    send, recv, recv_counts = counted_exchange(gb.partials_count, functools.partial(gb.partials_export, stage2=stage2),
                                               PA_PARTIAL_WORDS_STAGE2 if stage2 else PA_PARTIAL_WORDS)
    merged = adopt(MergedGroupBy(recv.data_ptr(), recv_counts, [a for a in aggs if a != "count_distinct"], value_format, key_format,
                                 device=dev.index, stream=stream))
    merged._keep = (send, recv)
    if distinct:
        _, precv, precv_counts = counted_exchange(gb.distinct_pairs_count, gb.distinct_pairs_export, PA_DISTINCT_PAIR_WORDS)
        merged.merge_distinct_pairs(precv.data_ptr(), precv_counts)
    return merged


def _sharded_utf8(gb, values, aggs, value_format, key_format, group, stream, dev, world):
    import torch
    import torch.distributed as dist
    from .groupby import MergedGroupBy, PaError
    stage2 = any(PA_AGG[a] & PA_AGG_STAGE2 for a in aggs)
    words = PA_PARTIAL_WORDS_STAGE2 if stage2 else PA_PARTIAL_WORDS
    # every seed is reached at most twice: by a shard's own check, and by a collision an owner saw
    for _ in range(2 * MAX_HASH_SEEDS):
        gb.aggregate(values, aggs, fetch=False)
        seed, unanimous = agree_key_hash_seed(gb, group)
        if not unanimous:
            continue
        counts, nbytes = gb.partials_count_utf8(world)
        send = torch.empty((max(sum(counts), 1), words), dtype=torch.int64, device=dev)
        lens = torch.empty(max(sum(counts), 1), dtype=torch.int32, device=dev)
        data = torch.empty(max(sum(nbytes), 1), dtype=torch.uint8, device=dev)
        gb.partials_export_utf8(world, send.data_ptr(), send.shape[0], lens.data_ptr(), data.data_ptr(), data.numel(), stage2=stage2)
        recv, recv_counts = exchange_records(send[:sum(counts)], counts, group, words=words)
        rlens, rdata, _, recv_bytes = exchange_key_strings(lens[:sum(counts)], data[:sum(nbytes)], counts, nbytes, group)
        torch.cuda.synchronize()
        merged = MergedGroupBy(recv.data_ptr(), recv_counts, [a for a in aggs if a != "count_distinct"], value_format, key_format,
                               device=dev.index, stream=stream)
        collided = merged.merge_key_strings(rlens.data_ptr(), rdata.data_ptr(), recv_counts, recv_bytes, [seed] * world)
        flag = torch.tensor([int(collided)], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=group)
        if int(flag.item()):
            merged.close()
            if seed + 1 >= MAX_HASH_SEEDS:
                raise PaError(4, "utf8 keys: four differently seeded 64-bit hashes all collided")
            gb.set_key_hash_seed(seed + 1)
            continue
        merged._keep = (send, recv)
        if "count_distinct" in aggs:
            counts = gb.distinct_pairs_count(world)
            psend = torch.empty((max(sum(counts), 1), PA_DISTINCT_PAIR_WORDS), dtype=torch.int64, device=dev)
            gb.distinct_pairs_export(world, psend.data_ptr(), psend.shape[0])
            precv, precv_counts = exchange_records(psend[:sum(counts)], counts, group, words=PA_DISTINCT_PAIR_WORDS)
            torch.cuda.synchronize()
            merged.merge_distinct_pairs(precv.data_ptr(), precv_counts)
        return merged
    raise PaError(4, "utf8 keys: four differently seeded 64-bit hashes all collided")


def resample_anchor(first_ts_local: Optional[int], ticks_per_day: int = 86_400 * 10**9, group=None) -> int:
    """Common bucket anchor for a row-range sharded resample (SURVEY §8e, last row): the reference anchors the
    bucket grid at the start of the day of the FIRST timestamp (TimeGrouperOrigin::StartDay, resample.cpp:85-178);
    every rank must use the global first timestamp, not its shard's.  Returns start_day(min over ranks) to pass as
    `origin="custom", origin_custom_ns=...`.  first_ts_local: this shard's first timestamp (None = empty shard)."""
    import torch
    import torch.distributed as dist
    big = (1 << 63) - 1
    t = torch.tensor([big if first_ts_local is None else int(first_ts_local)], dtype=torch.int64)
    if dist.get_backend(group) == "nccl":
        t = t.cuda()
    dist.all_reduce(t, op=dist.ReduceOp.MIN, group=group)
    first = int(t.item())
    if first == big:
        return 0
    return first - first % ticks_per_day          # (Python's % is a floor modulus: correct before the epoch too)


def gather_result(local: Dict[str, "np.ndarray"], first_rows: "np.ndarray", group=None) -> Dict[str, "np.ndarray"]:
    """All-gather the owners' result columns and restore global first-appearance order
    (stable sort by global first row).  Host-side convenience for tests / small results."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    parts: List = [None] * world
    dist.all_gather_object(parts, (local, first_rows), group=group)
    fr = np.concatenate([p[1] for p in parts])
    order = np.argsort(fr, kind="stable")
    return {k: np.concatenate([p[0][k] for p in parts])[order] for k in local}
