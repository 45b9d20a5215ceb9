"""Host-side harness over the C ABI, shaped like the reference's classes:

    pd::GroupBy   (/root/reference/src/group_by.h:22-247)    -> GroupBy
    pd::Resampler (/root/reference/src/group_by.h:255-299)   -> Resampler
    pd::resample  (/root/reference/src/resample.h:91-122)    -> resample()

Method names, argument meaning (a column name -> one array, a list of names -> one array per name
indexed by the unique keys) and error behaviour follow the reference.  Everything computes in
libpa_b200.so on the GPU; columns may be pyarrow arrays (host memory, copied by the library) or
DeviceColumn views of CUDA memory (zero copy).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence, Tuple, Union

import pyarrow as pa

from . import _lib
from ._lib import (ARROW_DEVICE_CPU, ARROW_DEVICE_CUDA, PA_AGG, ArrowArray, ArrowDeviceArray, ArrowSchema,
                   PaKeyLayout, PaOptions)

_RELEASE_ARRAY = C.CFUNCTYPE(None, C.POINTER(ArrowArray))
_RELEASE_SCHEMA = C.CFUNCTYPE(None, C.POINTER(ArrowSchema))
_PATHS = {"auto": 0, "lowcard": 1, "global": 2}
ORIGIN = {"epoch": 0, "start": 1, "start_day": 2, "end": 3, "end_day": 4, "custom": 5}


class PaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"[pa_b200 {code}] {msg}")
        self.code = code


def _check(rc):
    if rc != 0:
        raise PaError(rc, _lib.load().pa_last_error().decode())


class DeviceColumn:
    """A primitive Arrow column whose buffers live in CUDA memory (borrowed, not owned)."""

    def __init__(self, data_ptr: int, length: int, fmt: str, device_id: int = 0, valid_ptr: Optional[int] = None,
                 null_count: int = 0, offset: int = 0, keepalive=None):
        self.data_ptr, self.length, self.fmt, self.device_id = int(data_ptr), int(length), fmt, int(device_id)
        self.valid_ptr, self.null_count, self.offset = valid_ptr, int(null_count), int(offset)
        self.keepalive = keepalive

    @staticmethod
    def from_torch(t, fmt: Optional[str] = None, valid=None, null_count: int = 0) -> "DeviceColumn":
        import torch
        fmts = {torch.int64: "l", torch.float64: "g", torch.int32: "i", torch.float32: "f",
                torch.int16: "s", torch.int8: "c", torch.uint8: "C"}
        assert t.is_cuda and t.is_contiguous()
        return DeviceColumn(t.data_ptr(), t.numel(), fmt or fmts[t.dtype], t.device.index,
                            valid_ptr=None if valid is None else valid.data_ptr(), null_count=null_count,
                            keepalive=(t, valid))


class _Ingested:
    """Owner of the device buffers pa_column_to_device made (released when the last DeviceColumn drops it)."""

    def __init__(self, dev):
        self.dev = dev

    def __del__(self):
        try:
            if self.dev.array.release:
                _RELEASE_ARRAY(self.dev.array.release)(C.byref(self.dev.array))
        except Exception:
            pass


def to_device(array: pa.Array, device: Optional[int] = None, stream: Optional[int] = None) -> DeviceColumn:
    """Ingest: copy one host Arrow array (fixed-width numeric / temporal) to the device once (pa_column_to_device:
    pageable memory goes through the library's pinned staging pipeline) and use it in place from then on."""
    if isinstance(array, pa.ChunkedArray):
        array = array.combine_chunks()
    src = _CArg(array)
    out = ArrowDeviceArray()
    opt = _options(0, "auto", device, stream)
    try:
        _check(_lib.load().pa_column_to_device(C.byref(src.dev), C.byref(src.schema), C.byref(opt), C.byref(out)))
        fmt = src.schema.format.decode()
    finally:
        src.close()
    if out.array.n_buffers != 2:
        _RELEASE_ARRAY(out.array.release)(C.byref(out.array))
        raise PaError(3, "to_device(): primitive columns only in the Python harness")
    owner = _Ingested(out)
    return DeviceColumn(out.array.buffers[1], out.array.length, fmt, out.device_id, valid_ptr=out.array.buffers[0],
                        null_count=out.array.null_count, offset=out.array.offset, keepalive=owner)


class _CArg:
    """ArrowDeviceArray + ArrowSchema pair ready to pass to the library; releases exports on close."""

    def __init__(self, col):
        self.dev = ArrowDeviceArray()
        self.schema = ArrowSchema()
        self._exported = False
        self._keep = []
        if isinstance(col, DeviceColumn):
            bufs = (C.c_void_p * 2)(col.valid_ptr, col.data_ptr)
            fmt = C.c_char_p(col.fmt.encode())
            self._keep += [bufs, fmt, col.keepalive]
            a = self.dev.array
            a.length, a.null_count, a.offset, a.n_buffers, a.n_children = col.length, col.null_count, col.offset, 2, 0
            a.buffers = C.cast(bufs, C.POINTER(C.c_void_p))
            self.dev.device_id, self.dev.device_type = col.device_id, ARROW_DEVICE_CUDA
            self.schema.format = fmt
            self.schema.name = b""
            self.schema.flags = 2
        else:
            if isinstance(col, pa.ChunkedArray):
                col = col.combine_chunks()
            if not isinstance(col, pa.Array):
                col = pa.array(col)
            col._export_to_c(C.addressof(self.dev), C.addressof(self.schema))
            self._keep.append(col)
            self._exported = True
            self.dev.device_id, self.dev.device_type = -1, ARROW_DEVICE_CPU

    def close(self):
        if self._exported:
            if self.dev.array.release:
                _RELEASE_ARRAY(self.dev.array.release)(C.byref(self.dev.array))
            if self.schema.release:
                _RELEASE_SCHEMA(self.schema.release)(C.byref(self.schema))
            self._exported = False


def _pack_args(cols):
    args = [_CArg(c) for c in cols]
    devs = (ArrowDeviceArray * len(args))()
    schemas = (ArrowSchema * len(args))()
    for i, a in enumerate(args):
        C.memmove(C.addressof(devs[i]), C.addressof(a.dev), C.sizeof(ArrowDeviceArray))
        C.memmove(C.addressof(schemas[i]), C.addressof(a.schema), C.sizeof(ArrowSchema))
    return args, devs, schemas


def _import(out_a, out_s) -> pa.Array:
    return pa.Array._import_from_c(C.addressof(out_a), C.addressof(out_s))


def _options(expected_groups=0, path="auto", device=None, stream=None, row_base=0, no_dense=False,
             no_partition=False, bucket_bits=0, sm_reserve=0) -> PaOptions:
    o = PaOptions()
    _lib.load().pa_options_init(C.byref(o))
    o.expected_groups = int(expected_groups)
    o.row_base = int(row_base)
    o.path = _PATHS[path]
    o.lowcard_no_dense = 1 if no_dense else 0
    o.no_partition = 1 if no_partition else 0
    o.bucket_bits = int(bucket_bits)
    o.sm_reserve = int(sm_reserve)
    if device is not None:
        o.device = int(device)
    if stream is not None:
        o.cuda_stream = int(stream)
    return o


Column = Union[pa.Array, DeviceColumn]


class GroupBy:
    """pd::GroupBy: hash group-by on one or several (up to 4) key columns.

    `frame` maps column names to columns (pyarrow RecordBatch/Table, or a dict of pa.Array /
    DeviceColumn); `key` names the key column(s) — or pass key arrays directly with `key_arrays`
    (DataFrame::group_by(ArrayPtr), dataframe.cpp:1231-1235).

    A composite key that packs into 64 bits groups on its packed word; a wider one (two int64 ids, say) groups on a
    seeded 64-bit row hash that the first pass checks row by row.  encode_utf8=True dictionary-encodes utf8 members of
    a composite key on the host (their codes pack); encode_utf8=False hands them to the library as strings (a hashed
    key, unique(j) returns the strings).  Only packed composite keys cross GPUs or host chunks."""

    def __init__(self, key, frame=None, *, key_arrays: Optional[Sequence[Column]] = None, expected_groups: int = 0,
                 path: str = "auto", device: Optional[int] = None, stream: Optional[int] = None, row_base: int = 0,
                 no_dense: bool = False, no_partition: bool = False, bucket_bits: int = 0, sm_reserve: int = 0,
                 encode_utf8: bool = True, _handle=None):
        self._L = _lib.load()
        self._h = C.c_void_p()
        self._frame = self._as_dict(frame)
        self._dicts: List[Optional[pa.Array]] = []
        self._encode_utf8 = encode_utf8
        if _handle is not None:
            self._h = _handle
            self.key_names = ["__resampler_idx__"]
            self._dicts = [None]
            return
        self.key_names = [key] if isinstance(key, str) else list(key)
        if key_arrays is None:
            try:
                key_arrays = [self._frame[k] for k in self.key_names]
            except KeyError as e:
                raise RuntimeError(f"Invalid column: {e.args[0]}")   # std::runtime_error in the reference ctor
        key_arrays = [self._normalise_key(k) for k in key_arrays]
        args, devs, schemas = _pack_args(key_arrays)
        self._key_args = args          # keys are borrowed until destroy
        self.key_formats = [a.schema.format.decode() for a in args]   # (dictionary columns: the index format)
        opt = _options(expected_groups, path, device, stream, row_base, no_dense, no_partition, bucket_bits, sm_reserve)
        try:
            _check(self._L.pa_groupby_create(devs, schemas, len(args), C.byref(opt), C.byref(self._h)))
        except Exception:
            for a in args:
                a.close()
            raise

    def _normalise_key(self, k):
        if isinstance(k, pa.ChunkedArray):
            k = k.combine_chunks()
        if (isinstance(k, pa.Array) and (pa.types.is_string(k.type) or pa.types.is_large_string(k.type))
                and len(self.key_names) > 1 and self._encode_utf8):
            # a utf8 column inside a COMPOSITE key is dictionary-encoded (its codes pack into the 64-bit key); a single
            # utf8 key, or any with encode_utf8=False, goes to the device as strings (format "u": offsets + bytes,
            # csrc/strkeys.cuh, csrc/rowkeys.cuh)
            k = k.dictionary_encode()
        self._dicts.append(k.dictionary if isinstance(k, pa.DictionaryArray) else None)
        return k

    @staticmethod
    def _as_dict(frame) -> Dict[str, Column]:
        if frame is None:
            return {}
        if isinstance(frame, (pa.RecordBatch, pa.Table)):
            return {n: frame.column(n) for n in frame.schema.names}
        return dict(frame)

    # ---- lifetime ----
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._L.pa_groupby_destroy(self._h)
            self._h = C.c_void_p()
            for a in getattr(self, "_key_args", []):
                a.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- group_by.h:33-60 ----
    def groupSize(self) -> int:
        n = C.c_int64()
        _check(self._L.pa_groupby_num_groups(self._h, C.byref(n)))
        return n.value

    num_groups = property(groupSize)

    def unique(self, key_i: int = 0) -> pa.Array:
        a, s = ArrowArray(), ArrowSchema()
        _check(self._L.pa_groupby_unique(self._h, key_i, C.byref(a), C.byref(s)))
        out = _import(a, s)
        d = self._dicts[key_i] if key_i < len(self._dicts) else None
        if d is not None:
            out = pa.DictionaryArray.from_arrays(out, d)
        return out

    def key_layout(self) -> PaKeyLayout:
        """pa_groupby_key_layout: how this composite key packs into 64 bits (with its dictionaries' fingerprints)."""
        out = PaKeyLayout()
        _check(self._L.pa_groupby_key_layout(self._h, C.byref(out)))
        return out

    def set_key_layout(self, layout: PaKeyLayout):
        """pa_groupby_set_key_layout: repack the composite key under `layout` (one that all shards agreed on, see
        distributed.agree_key_layout); groups and results of earlier aggregates are dropped."""
        _check(self._L.pa_groupby_set_key_layout(self._h, C.byref(layout)))

    def first_rows(self) -> pa.Array:
        """Global row number of the first row of every group (result order)."""
        a, s = ArrowArray(), ArrowSchema()
        _check(self._L.pa_groupby_first_rows(self._h, C.byref(a), C.byref(s)))
        return _import(a, s)

    # ---- aggregation core ----
    def aggregate(self, values: Column, aggs: Sequence[str], fetch: bool = True, wait: bool = True) -> Dict[str, pa.Array]:
        """One fused pass computing `aggs` of `values` per group.  wait=False (device-resident inputs): queue the
        pass and return; the next call that needs the result (fetch, groupSize, timing, ...) completes it."""
        mask = 0
        for a in aggs:
            mask |= PA_AGG[a]
        arg = _CArg(values)
        deferred = not (wait or fetch)
        fn = self._L.pa_groupby_aggregate_async if deferred else self._L.pa_groupby_aggregate
        try:
            _check(fn(self._h, C.byref(arg.dev), C.byref(arg.schema), mask))
        finally:
            if deferred:
                # the handle keeps borrowed pointers of the value column until the pass is finished (a declined
                # dense pass is redone from them): keep the column alive until the next call replaces it
                self._pending_arg = arg
            else:
                arg.close()
                self._pending_arg = None
        if not fetch:
            return {}
        return {a: self.fetch(a) for a in aggs}

    def fetch(self, agg: str) -> pa.Array:
        a, s = ArrowArray(), ArrowSchema()
        _check(self._L.pa_groupby_fetch(self._h, PA_AGG[agg], C.byref(a), C.byref(s)))
        return _import(a, s)

    def sync(self):
        _check(self._L.pa_groupby_sync(self._h))

    def row_ids(self) -> pa.Array:
        """Grouper::Consume equivalent (dataframe.cpp:1584): uint32 group id of every row, ids numbered in
        first-appearance order (= positions in unique())."""
        out_a, out_s = ArrowArray(), ArrowSchema()
        _check(self._L.pa_groupby_row_ids(self._h, C.byref(out_a), C.byref(out_s)))
        return _import(out_a, out_s)

    def groupings(self, rows: bool = True):
        """Grouper::MakeGroupings equivalent (dataframe.cpp:1586-1588): (offsets int32[G+1], rows int32[n]) — group j
        owns rows[offsets[j]:offsets[j+1]], ascending.  rows=False: offsets only."""
        oa, os_, ra, rs = ArrowArray(), ArrowSchema(), ArrowArray(), ArrowSchema()
        if rows:
            _check(self._L.pa_groupby_groupings(self._h, C.byref(oa), C.byref(os_), C.byref(ra), C.byref(rs)))
            return _import(oa, os_), _import(ra, rs)
        _check(self._L.pa_groupby_groupings(self._h, C.byref(oa), C.byref(os_), None, None))
        return _import(oa, os_), None

    def take_grouped(self, column: Column) -> pa.Array:
        """Grouper::ApplyGroupings equivalent for one column (dataframe.cpp:1546,1562): the column gathered on the
        device into group-contiguous order (see groupings())."""
        arg = _CArg(column)
        a, s = ArrowArray(), ArrowSchema()
        try:
            _check(self._L.pa_groupby_take_grouped(self._h, C.byref(arg.dev), C.byref(arg.schema), C.byref(a), C.byref(s)))
        finally:
            arg.close()
        return _import(a, s)

    def groupings_timing(self) -> dict:
        b, t = C.c_double(), C.c_double()
        _check(self._L.pa_groupby_groupings_timing(self._h, C.byref(b), C.byref(t)))
        return {"build_ms": b.value, "take_ms": t.value}

    # ---- multi-GPU: hash-partitioned partial aggregates (include/pa_b200.h, SURVEY §8e) ----
    def partials_count(self, n_parts: int) -> List[int]:
        counts = (C.c_int64 * n_parts)()
        _check(self._L.pa_groupby_partials_count(self._h, n_parts, counts))
        return list(counts)

    def partials_export(self, n_parts: int, records_ptr: int, capacity_records: int, stage2: bool = False):
        """stage2=True: PA_PARTIAL_WORDS_STAGE2-word records that also carry the product / variance terms of the last
        aggregate (which must have computed product, variance or stddev); else PA_PARTIAL_WORDS-word records."""
        fn = self._L.pa_groupby_partials_export_stage2 if stage2 else self._L.pa_groupby_partials_export
        _check(fn(self._h, n_parts, records_ptr, capacity_records))

    # ---- a single utf8 / large_utf8 key across shards: records travel with their key bytes ----
    def key_hash_seed(self) -> int:
        """pa_groupby_key_hash_seed: the seed this utf8 key, or hashed composite key, is hashed with (raised by the
        handle's own check)."""
        out = C.c_uint64()
        _check(self._L.pa_groupby_key_hash_seed(self._h, C.byref(out)))
        return out.value

    def set_key_hash_seed(self, seed: int):
        """pa_groupby_set_key_hash_seed: re-hash the key with `seed` (one that all shards agreed on, see
        distributed.agree_key_hash_seed); groups and results of earlier aggregates are dropped."""
        _check(self._L.pa_groupby_set_key_hash_seed(self._h, int(seed)))

    def partials_count_utf8(self, n_parts: int) -> Tuple[List[int], List[int]]:
        """Records and key bytes owned by each of n_parts ranks (after an aggregate)."""
        recs, nbytes = (C.c_int64 * n_parts)(), (C.c_int64 * n_parts)()
        _check(self._L.pa_groupby_partials_count_utf8(self._h, n_parts, recs, nbytes))
        return list(recs), list(nbytes)

    def partials_export_utf8(self, n_parts: int, records_ptr: int, capacity_records: int, lengths_ptr: int, bytes_ptr: int,
                             capacity_bytes: int, stage2: bool = False):
        """Records (as partials_export), one uint32 key length per record and the key bytes, grouped by owner in the same
        order, into device memory (after partials_count_utf8)."""
        _check(self._L.pa_groupby_partials_export_utf8(self._h, n_parts, int(bool(stage2)), records_ptr, capacity_records,
                                                       lengths_ptr, bytes_ptr, capacity_bytes))

    def partials_export_padded(self, n_parts: int, blocks_ptr: int, block_records: int):
        _check(self._L.pa_groupby_partials_export_padded(self._h, n_parts, blocks_ptr, block_records))

    def distinct_pairs_count(self, n_parts: int) -> List[int]:
        """count_distinct across shards: this handle's distinct (key, value) pairs owned by each of n_parts ranks (the
        last aggregate must have computed count_distinct)."""
        counts = (C.c_int64 * n_parts)()
        _check(self._L.pa_groupby_distinct_pairs_count(self._h, n_parts, counts))
        return list(counts)

    def distinct_pairs_export(self, n_parts: int, pairs_ptr: int, capacity_pairs: int):
        """PA_DISTINCT_PAIR_WORDS-word pair records, grouped by owner, into device memory (after distinct_pairs_count)."""
        _check(self._L.pa_groupby_distinct_pairs_export(self._h, n_parts, pairs_ptr, capacity_pairs))

    def timing(self) -> dict:
        total = C.c_double()
        st = (C.c_double * 4)()
        _check(self._L.pa_groupby_last_timing(self._h, C.byref(total), st))
        path, launches = C.c_int32(), C.c_int32()
        _check(self._L.pa_groupby_last_path(self._h, C.byref(path), C.byref(launches)))
        det = (C.c_int32 * 4)()
        _check(self._L.pa_groupby_last_detail(self._h, det))
        return {"total_ms": total.value, "pack_ms": st[0], "scan_ms": st[1], "merge_ms": st[2], "emit_ms": st[3],
                "path": {1: "lowcard", 2: "global", 3: "resample"}.get(path.value, "?"), "launches": launches.value,
                "mode": {0: None, 1: "dense", 2: "hash", 3: "smem-front", 4: "partitioned", 5: "bucketed",
                         6: "dense-known"}.get(det[0]), "replication": 1 << det[1], "passes": det[2]}

    # ---- the reference's method surface (group_by.h:85-139): name -> array, [names] -> {name: array} ----
    def _agg(self, agg: str, arg):
        if isinstance(arg, str):
            return self.aggregate(self._column(arg), [agg])[agg]
        if isinstance(arg, (list, tuple)):
            return {name: self.aggregate(self._column(name), [agg])[agg] for name in arg}
        return self.aggregate(arg, [agg])[agg]        # a column object

    def _column(self, name: str):
        try:
            return self._frame[name]
        except KeyError:
            raise RuntimeError(f"Invalid column: {name}")

    def sum(self, arg): return self._agg("sum", arg)
    def mean(self, arg): return self._agg("mean", arg)
    def count(self, arg): return self._agg("count", arg)
    def min(self, arg): return self._agg("min", arg)
    def max(self, arg): return self._agg("max", arg)
    def first(self, arg): return self._agg("first", arg)
    def last(self, arg): return self._agg("last", arg)
    # second-stage aggregates (group_by.h:88-136 / dataframe.cpp:1516-1536): one extra pass over keys + values
    def product(self, arg): return self._agg("product", arg)
    def variance(self, arg): return self._agg("variance", arg)
    def stddev(self, arg): return self._agg("stddev", arg)
    # boolean columns (GROUPBY_NUMERIC_AGG(all|any, bool), dataframe.cpp:1522-1524)
    def all(self, arg): return self._agg("all", arg)
    def any(self, arg): return self._agg("any", arg)
    def count_distinct(self, arg): return self._agg("count_distinct", arg)     # dataframe.cpp:1528; sort based

    def min_max(self, arg):
        """GroupBy::min_max (dataframe.cpp:1602-1696): one pass, two columns."""
        if isinstance(arg, str):
            r = self.aggregate(self._column(arg), ["min", "max"])
            return {"min": r["min"], "max": r["max"]}
        out = {}
        for name in arg:
            r = self.aggregate(self._column(name), ["min", "max"])
            out[name + "_min"], out[name + "_max"] = r["min"], r["max"]
        return out


class MergedGroupBy(GroupBy):
    """Owner-side result of the multi-GPU merge: the groups whose hash(key) % world == rank."""

    def __init__(self, records_ptr: int, counts_by_source: Sequence[int], aggs: Sequence[str], value_format: str,
                 key_format: str, device: Optional[int] = None, stream: Optional[int] = None,
                 padded_block_records: int = 0):
        """counts_by_source: per-source record counts (counted exchange), or — with padded_block_records > 0 —
        just the number of sources as a list of that length (padded exchange, counts live in the block headers)."""
        self._L = _lib.load()
        self._h = C.c_void_p()
        self._frame, self._dicts, self.key_names, self._key_args = {}, [None], ["key"], []
        mask = 0
        for a in aggs:
            mask |= PA_AGG[a]
        opt = _options(0, "auto", device, stream)
        if padded_block_records > 0:
            _check(self._L.pa_merge_create_padded(records_ptr, len(counts_by_source), padded_block_records, mask,
                                                  value_format.encode(), key_format.encode(), C.byref(opt), C.byref(self._h)))
            return
        counts = (C.c_int64 * len(counts_by_source))(*[int(c) for c in counts_by_source])
        _check(self._L.pa_merge_create(records_ptr, counts, len(counts_by_source), mask, value_format.encode(),
                                       key_format.encode(), C.byref(opt), C.byref(self._h)))

    def set_composite_key(self, layout: PaKeyLayout, key_formats: Sequence[str], key_names: Optional[Sequence[str]] = None,
                          dictionaries: Optional[Sequence[Optional[pa.Array]]] = None):
        """pa_merge_set_key_layout: the records were merged by their packed composite key (key format "L"); unique(j)
        then returns key column j (`key_formats[j]`: a dictionary column's index format, wrapped with
        dictionaries[j])."""
        fmts = (C.c_char_p * len(key_formats))(*[f.encode() for f in key_formats])
        _check(self._L.pa_merge_set_key_layout(self._h, C.byref(layout), fmts))
        self._adopt_keys(key_names or [f"key{j}" for j in range(len(key_formats))], dictionaries or [None] * len(key_formats))

    def _adopt_keys(self, key_names, dictionaries):
        self.key_names, self._dicts = list(key_names), list(dictionaries)

    def merge_key_strings(self, lengths_ptr: int, bytes_ptr: int, records_by_source: Sequence[int], bytes_by_source: Sequence[int],
                          seed_by_source: Sequence[int]) -> bool:
        """pa_merge_key_strings (key format "u" / "U"): attaches the merged groups' key strings from the received lengths and
        bytes, grouped by source.  Returns True when two different strings shared a hash: then nothing is attached and
        the ranks retry with the next seed.  The record buffer given to the constructor must still be alive."""
        n = len(records_by_source)
        recs = (C.c_int64 * n)(*[int(c) for c in records_by_source])
        nbytes = (C.c_int64 * n)(*[int(c) for c in bytes_by_source])
        seeds = (C.c_uint64 * n)(*[int(c) for c in seed_by_source])
        collided = C.c_int32()
        _check(self._L.pa_merge_key_strings(self._h, lengths_ptr, bytes_ptr, recs, nbytes, seeds, n, C.byref(collided)))
        return bool(collided.value)

    def merge_distinct_pairs(self, pairs_ptr: int, counts_by_source: Sequence[int]):
        """Adds count_distinct (fetch("count_distinct")) from the received distinct-pair records, grouped by source."""
        counts = (C.c_int64 * len(counts_by_source))(*[int(c) for c in counts_by_source])
        _check(self._L.pa_merge_distinct_pairs(self._h, pairs_ptr, counts, len(counts_by_source)))


def _merged_from_handle(h) -> "MergedGroupBy":
    m = MergedGroupBy.__new__(MergedGroupBy)
    m._L = _lib.load()
    m._h = h
    m._frame, m._dicts, m.key_names, m._key_args = {}, [None], ["key"], []
    return m


MergedGroupBy._from_handle = staticmethod(_merged_from_handle)


def aggregate_chunked(keys, values: pa.Array, aggs: Sequence[str], chunk_rows: int, *, device: Optional[int] = None,
                      row_base: int = 0) -> "MergedGroupBy":
    """Host columns larger than the device (or than 2^32-2 rows): pa_groupby_aggregate_chunked — the columns are
    aggregated `chunk_rows` rows at a time and the chunks' partial records merged like ranks'.  `keys`: one key array,
    or a list of them (a composite key: utf8 members are dictionary-encoded once over the whole column; unique(j)
    returns a DictionaryArray for dictionary columns).  A single utf8 / large_utf8 key stays strings: its key bytes
    travel with the chunks' records and unique() returns the input's string type."""
    mask = 0
    for a in aggs:
        mask |= PA_AGG[a]
    composite = isinstance(keys, (list, tuple))
    key_list = list(keys) if composite else [keys]
    if composite:
        key_list = [k.combine_chunks() if isinstance(k, pa.ChunkedArray) else k for k in key_list]
        key_list = [k.dictionary_encode() if isinstance(k, pa.Array) and (pa.types.is_string(k.type) or pa.types.is_large_string(k.type))
                    else k for k in key_list]
    args, devs, schemas = _pack_args(key_list)
    va = _CArg(values)
    h = C.c_void_p()
    opt = _options(0, "auto", device, None, row_base=row_base)
    try:
        _check(_lib.load().pa_groupby_aggregate_chunked_keys(devs, schemas, len(args), C.byref(va.dev), C.byref(va.schema),
                                                             mask, int(chunk_rows), C.byref(opt), C.byref(h)))
    finally:
        for a in args:
            a.close()
        va.close()
    m = MergedGroupBy._from_handle(h)
    if composite:
        m._adopt_keys([f"key{j}" for j in range(len(key_list))],
                      [k.dictionary if isinstance(k, pa.DictionaryArray) else None for k in key_list])
    return m


class Resampler(GroupBy):
    """pd::Resampler (group_by.h:255-299): every aggregate runs over all columns of the frame and
    the result is indexed by the bucket labels (`index()`)."""

    def index(self) -> pa.Array:
        return self.unique()

    def data(self):
        return self._frame

    def _all(self, agg):
        return {name: self.aggregate(col, [agg])[agg] for name, col in self._frame.items()}

    def sum(self, arg=None): return self._all("sum") if arg is None else super().sum(arg)
    def mean(self, arg=None): return self._all("mean") if arg is None else super().mean(arg)
    def count(self, arg=None): return self._all("count") if arg is None else super().count(arg)
    def min(self, arg=None): return self._all("min") if arg is None else super().min(arg)
    def max(self, arg=None): return self._all("max") if arg is None else super().max(arg)
    def first(self, arg=None): return self._all("first") if arg is None else super().first(arg)
    def last(self, arg=None): return self._all("last") if arg is None else super().last(arg)
    def product(self, arg=None): return self._all("product") if arg is None else super().product(arg)
    def variance(self, arg=None): return self._all("variance") if arg is None else super().variance(arg)
    def stddev(self, arg=None): return self._all("stddev") if arg is None else super().stddev(arg)


def resample(frame, index: Column, freq_ns: int, closed_right: bool = False, label_right: bool = False,
             origin: str = "start_day", origin_custom_ns: int = 0, offset_ns: int = 0, *, device=None,
             stream=None, row_base: int = 0) -> Resampler:
    """pd::resample(df, time_duration rule, ...) (resample.h:91-122) on a sorted timestamp index.
    row_base: global row number of local row 0 (multi-GPU row-range shards; use a common `origin="custom"` anchor on
    every rank — distributed.resample_anchor — so that all shards cut the same bucket grid)."""
    L = _lib.load()
    arg = _CArg(index)
    h = C.c_void_p()
    opt = _options(0, "auto", device, stream, row_base=row_base)
    try:
        _check(L.pa_resample_create(C.byref(arg.dev), C.byref(arg.schema), int(freq_ns), int(closed_right),
                                    int(label_right), ORIGIN[origin], int(origin_custom_ns), int(offset_ns),
                                    C.byref(opt), C.byref(h)))
    except Exception:
        arg.close()
        raise
    r = Resampler(None, frame, _handle=h)
    r._key_args = [arg]
    return r


# DateOffset::Type (core.h:122-134) by rule code (DateOffset::FromString, core.cpp:62-108)
OFFSET_TYPES = {"D": 0, "M": 1, "QS": 2, "Q": 3, "WS": 4, "W": 5, "MS": 6, "Y": 7, "YS": 8}


def resample_calendar(frame, index: Column, rule: str, closed_right: bool = False, label_right: bool = False, *,
                      device=None, stream=None) -> Resampler:
    """pd::resample(df, "<k><code>", ...) with a DateOffset rule (resample.h:62-88 -> resample.cpp:248-267): D, WS, MS,
    QS, YS; the month / quarter / week / year END codes and closed_right=False fail like the reference."""
    import re
    m = re.fullmatch(r"(\d*)([A-Za-z]+)", rule)
    if not m or m.group(2) not in OFFSET_TYPES:
        raise RuntimeError(f"Invalid time offset {rule}")
    mult = int(m.group(1)) if m.group(1) else 1
    L = _lib.load()
    arg = _CArg(index)
    h = C.c_void_p()
    opt = _options(0, "auto", device, stream)
    try:
        _check(L.pa_resample_create_calendar(C.byref(arg.dev), C.byref(arg.schema), OFFSET_TYPES[m.group(2)], mult,
                                             int(closed_right), int(label_right), C.byref(opt), C.byref(h)))
    except Exception:
        arg.close()
        raise
    r = Resampler(None, frame, _handle=h)
    r._key_args = [arg]
    return r


def downsample(frame, index: Column, rule: str, closed_label_right: bool = True, week_starts_monday: bool = True,
               start_epoch: bool = True, *, device=None, stream=None) -> Resampler:
    """DataFrame::downsample (dataframe.cpp:1265-1290): rule = "<multiple><unit>" with unit in N U L S T H D W M Q Y;
    labels = Floor/CeilTemporal(index) computed on the device (minus one day for W / M / Q / Y, as the reference)."""
    import re
    m = re.fullmatch(r"(\d*)([A-Za-z]+)", rule)
    if not m:
        raise RuntimeError(f"Invalid time offset {rule}")
    mult = int(m.group(1)) if m.group(1) else 1
    L = _lib.load()
    arg = _CArg(index)
    h = C.c_void_p()
    opt = _options(0, "auto", device, stream)
    try:
        _check(L.pa_downsample_create(C.byref(arg.dev), C.byref(arg.schema), mult, m.group(2)[0].encode(), int(closed_label_right),
                                      int(week_starts_monday), int(start_epoch), C.byref(opt), C.byref(h)))
    except Exception:
        arg.close()
        raise
    r = Resampler(None, frame, _handle=h)
    r._key_args = [arg]
    return r


class Sorted:
    """Stable argsort of one column on the device (pa_sort_create): what Series::argsort / Series::sort /
    DataFrame::sort_index get from arrow's array_sort_indices + Take (series.cpp:864-868,978-992,
    dataframe.cpp:1062-1071).  indices(): the uint64 sort indices; take(column): a column in sorted order."""

    def __init__(self, column: Column, ascending: bool = True, *, device: Optional[int] = None, stream: Optional[int] = None):
        self._L = _lib.load()
        self._h = C.c_void_p()
        arg = _CArg(column)
        opt = _options(0, "auto", device, stream)
        try:
            _check(self._L.pa_sort_create(C.byref(arg.dev), C.byref(arg.schema), int(bool(ascending)), C.byref(opt), C.byref(self._h)))
        finally:
            arg.close()

    def indices(self) -> pa.Array:
        a, s = ArrowArray(), ArrowSchema()
        _check(self._L.pa_sort_indices(self._h, C.byref(a), C.byref(s)))
        return _import(a, s)

    def take(self, column: Column) -> pa.Array:
        arg = _CArg(column)
        a, s = ArrowArray(), ArrowSchema()
        try:
            _check(self._L.pa_groupby_take_grouped(self._h, C.byref(arg.dev), C.byref(arg.schema), C.byref(a), C.byref(s)))
        finally:
            arg.close()
        return _import(a, s)

    def timing(self) -> dict:
        b, t = C.c_double(), C.c_double()
        _check(self._L.pa_groupby_groupings_timing(self._h, C.byref(b), C.byref(t)))
        return {"sort_ms": b.value, "take_ms": t.value}

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._L.pa_groupby_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class synth:
    """Device-side synthetic workload (SURVEY.md §8d); mirrors bench.py's host generator."""
    SEED_K, SEED_V, SEED_N, SEED_T = 42, 1337, 7, 99
    T0_NS = 1577836800 * 10**9

    @staticmethod
    def keys(t, n_groups: int, first_row: int = 0, seed: int = SEED_K):
        _check(_lib.load().pa_synth_keys_i64(t.data_ptr(), t.numel(), first_row, n_groups, seed, None))

    @staticmethod
    def vals(t, first_row: int = 0, seed: int = SEED_V):
        _check(_lib.load().pa_synth_vals_f64(t.data_ptr(), t.numel(), first_row, seed, None))

    @staticmethod
    def validity(t, n_rows: int, first_row: int = 0, seed: int = SEED_N, null_every: int = 10):
        _check(_lib.load().pa_synth_validity(t.data_ptr(), n_rows, first_row, seed, null_every, None))

    @staticmethod
    def timestamps(t, first_row: int = 0, t0_ns: int = T0_NS, step_ns: int = 60_000_000, seed: int = SEED_T):
        _check(_lib.load().pa_synth_timestamps(t.data_ptr(), t.numel(), first_row, t0_ns, step_ns, seed, None))
