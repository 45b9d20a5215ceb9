"""ctypes binding of libpa_b200.so (include/pa_b200.h).  Loading fails loudly: there is no
fallback implementation anywhere in this package."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PA_B200_LIB") or os.path.join(HERE, "lib", "libpa_b200.so")   # (override: kernel A/B experiments)

ARROW_DEVICE_CPU = 1
ARROW_DEVICE_CUDA = 2

PA_AGG = {"sum": 1, "mean": 2, "count": 4, "min": 8, "max": 16, "first": 32, "last": 64,
          "product": 128, "variance": 256, "stddev": 512, "all": 1024, "any": 2048, "count_distinct": 4096}
PA_PATH_AUTO, PA_PATH_LOWCARD, PA_PATH_GLOBAL = 0, 1, 2
PA_PARTIAL_WORDS = 11
PA_PARTIAL_WORDS_STAGE2 = 13   # records that also carry the product / variance terms
PA_AGG_STAGE2 = 128 | 256 | 512
PA_DISTINCT_PAIR_WORDS = 3     # count_distinct across shards: (key, value bits, flags) records
PA_MAX_KEY_COLS = 4

# every symbol include/pa_b200.h declares
EXPORTS = [
    "pa_last_error", "pa_version", "pa_options_init", "pa_device_count", "pa_groupby_create",
    "pa_groupby_num_groups", "pa_groupby_unique", "pa_groupby_aggregate", "pa_groupby_aggregate_async",
    "pa_groupby_fetch", "pa_column_aggregate",
    "pa_groupby_row_ids", "pa_groupby_groupings", "pa_groupby_take_grouped", "pa_groupby_groupings_timing", "pa_groupby_last_timing", "pa_groupby_last_path", "pa_groupby_last_detail",
    "pa_groupby_sync",
    "pa_groupby_destroy", "pa_column_to_device", "pa_sort_create", "pa_sort_indices", "pa_resample_create", "pa_resample_create_calendar", "pa_downsample_create", "pa_groupby_partials_count", "pa_groupby_partials_export",
    "pa_groupby_partials_export_stage2",
    "pa_groupby_distinct_pairs_count", "pa_groupby_distinct_pairs_export", "pa_merge_distinct_pairs",
    "pa_merge_create", "pa_groupby_aggregate_chunked", "pa_groupby_partials_export_padded", "pa_merge_create_padded", "pa_groupby_first_rows", "pa_synth_keys_i64", "pa_synth_vals_f64",
    "pa_synth_validity", "pa_synth_timestamps",
    "pa_comm_unique_id", "pa_comm_create", "pa_comm_adopt", "pa_comm_destroy", "pa_groupby_sharded_aggregate", "pa_comm_last_phases", "pa_comm_last_exchange",
    "pa_comm_last_distinct",
    "pa_groupby_key_layout", "pa_key_layout_agree", "pa_groupby_set_key_layout", "pa_merge_set_key_layout",
    "pa_groupby_aggregate_chunked_keys", "pa_comm_last_key_layout",
    "pa_groupby_key_hash_seed", "pa_groupby_set_key_hash_seed", "pa_groupby_partials_count_utf8", "pa_groupby_partials_export_utf8",
    "pa_merge_key_strings", "pa_comm_last_key_strings",
]


class ArrowSchema(C.Structure):
    pass


ArrowSchema._fields_ = [("format", C.c_char_p), ("name", C.c_char_p), ("metadata", C.c_char_p),
                        ("flags", C.c_int64), ("n_children", C.c_int64),
                        ("children", C.POINTER(C.POINTER(ArrowSchema))), ("dictionary", C.POINTER(ArrowSchema)),
                        ("release", C.c_void_p), ("private_data", C.c_void_p)]


class ArrowArray(C.Structure):
    pass


ArrowArray._fields_ = [("length", C.c_int64), ("null_count", C.c_int64), ("offset", C.c_int64),
                       ("n_buffers", C.c_int64), ("n_children", C.c_int64), ("buffers", C.POINTER(C.c_void_p)),
                       ("children", C.POINTER(C.POINTER(ArrowArray))), ("dictionary", C.POINTER(ArrowArray)),
                       ("release", C.c_void_p), ("private_data", C.c_void_p)]


class ArrowDeviceArray(C.Structure):
    _fields_ = [("array", ArrowArray), ("device_id", C.c_int64), ("device_type", C.c_int32),
                ("sync_event", C.c_void_p), ("reserved", C.c_int64 * 3)]


class PaOptions(C.Structure):
    _fields_ = [("device", C.c_int32), ("path", C.c_int32), ("expected_groups", C.c_int64),
                ("cuda_stream", C.c_void_p), ("row_base", C.c_int64), ("lowcard_no_dense", C.c_int64),
                ("no_partition", C.c_int64), ("bucket_bits", C.c_int64), ("sm_reserve", C.c_int64)]


class PaKeyLayout(C.Structure):
    """pa_key_layout: how a composite key packs into one 64-bit word (include/pa_b200.h)."""
    _fields_ = [("n_keys", C.c_int32), ("width", C.c_int32 * PA_MAX_KEY_COLS), ("bits", C.c_int32 * PA_MAX_KEY_COLS),
                ("nullable", C.c_int32 * PA_MAX_KEY_COLS), ("dict_fingerprint", C.c_uint64 * PA_MAX_KEY_COLS)]


_lib = None


def _preload_nccl():
    """libpa_b200.so needs libnccl.so.2 (pa_comm_*).  A process that also imports torch must end up with ONE copy, and
    torch wants the one bundled in its wheel set (newer than the system's): load that first, by path, when it exists,
    so that both resolve the soname to it whatever the import order."""
    import importlib.util
    try:
        spec = importlib.util.find_spec("nvidia")
    except (ImportError, ValueError):
        spec = None
    for base in (list(spec.submodule_search_locations) if spec and spec.submodule_search_locations else []):
        cand = os.path.join(base, "nccl", "lib", "libnccl.so.2")
        if os.path.exists(cand):
            C.CDLL(cand, mode=C.RTLD_GLOBAL)
            return


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"pandasarrow_b200: CUDA library {LIB_PATH} is missing. Build it with "
            "`python -m pandasarrow_b200.build` (nvcc, sm_100a). There is no CPU fallback.")
    _preload_nccl()
    L = C.CDLL(LIB_PATH)
    for name in EXPORTS:
        if not hasattr(L, name):
            raise ImportError(f"pandasarrow_b200: {LIB_PATH} does not export {name}")
    P = C.c_void_p
    L.pa_last_error.restype = C.c_char_p
    L.pa_options_init.argtypes = [C.POINTER(PaOptions)]
    L.pa_device_count.argtypes = [C.POINTER(C.c_int)]
    L.pa_groupby_create.argtypes = [C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema), C.c_int32,
                                    C.POINTER(PaOptions), C.POINTER(P)]
    L.pa_groupby_num_groups.argtypes = [P, C.POINTER(C.c_int64)]
    L.pa_groupby_unique.argtypes = [P, C.c_int32, C.POINTER(ArrowArray), C.POINTER(ArrowSchema)]
    L.pa_groupby_aggregate.argtypes = [P, C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema), C.c_uint32]
    L.pa_groupby_aggregate_async.argtypes = [P, C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema), C.c_uint32]
    L.pa_column_aggregate.argtypes = [C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema), C.c_uint32, C.c_int32,
                                      C.POINTER(PaOptions), C.POINTER(P)]
    L.pa_groupby_fetch.argtypes = [P, C.c_uint32, C.POINTER(ArrowArray), C.POINTER(ArrowSchema)]
    L.pa_groupby_first_rows.argtypes = [P, C.POINTER(ArrowArray), C.POINTER(ArrowSchema)]
    L.pa_groupby_row_ids.argtypes = [P, C.POINTER(ArrowArray), C.POINTER(ArrowSchema)]
    L.pa_groupby_groupings.argtypes = [P, C.POINTER(ArrowArray), C.POINTER(ArrowSchema), C.POINTER(ArrowArray), C.POINTER(ArrowSchema)]
    L.pa_groupby_take_grouped.argtypes = [P, C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema), C.POINTER(ArrowArray), C.POINTER(ArrowSchema)]
    L.pa_groupby_groupings_timing.argtypes = [P, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.pa_groupby_last_timing.argtypes = [P, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.pa_groupby_last_path.argtypes = [P, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    L.pa_groupby_last_detail.argtypes = [P, C.POINTER(C.c_int32)]
    L.pa_groupby_sync.argtypes = [P]
    L.pa_groupby_destroy.argtypes = [P]
    L.pa_groupby_destroy.restype = None
    L.pa_resample_create.argtypes = [C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema), C.c_int64, C.c_int32,
                                     C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.POINTER(PaOptions), C.POINTER(P)]
    L.pa_column_to_device.argtypes = [C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema), C.POINTER(PaOptions), C.POINTER(ArrowDeviceArray)]
    L.pa_sort_create.argtypes = [C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema), C.c_int32, C.POINTER(PaOptions), C.POINTER(P)]
    L.pa_sort_indices.argtypes = [P, C.POINTER(ArrowArray), C.POINTER(ArrowSchema)]
    L.pa_resample_create_calendar.argtypes = [C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema), C.c_int32, C.c_int32,
                                              C.c_int32, C.c_int32, C.POINTER(PaOptions), C.POINTER(P)]
    L.pa_downsample_create.argtypes = [C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema), C.c_int32, C.c_char, C.c_int32,
                                       C.c_int32, C.c_int32, C.POINTER(PaOptions), C.POINTER(P)]
    L.pa_groupby_partials_count.argtypes = [P, C.c_int32, C.POINTER(C.c_int64)]
    L.pa_groupby_partials_export.argtypes = [P, C.c_int32, P, C.c_int64]
    L.pa_groupby_partials_export_stage2.argtypes = [P, C.c_int32, P, C.c_int64]
    L.pa_groupby_distinct_pairs_count.argtypes = [P, C.c_int32, C.POINTER(C.c_int64)]
    L.pa_groupby_distinct_pairs_export.argtypes = [P, C.c_int32, P, C.c_int64]
    L.pa_merge_distinct_pairs.argtypes = [P, P, C.POINTER(C.c_int64), C.c_int32]
    L.pa_merge_create.argtypes = [P, C.POINTER(C.c_int64), C.c_int32, C.c_uint32, C.c_char_p, C.c_char_p,
                                  C.POINTER(PaOptions), C.POINTER(P)]
    L.pa_groupby_aggregate_chunked.argtypes = [C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema), C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema),
                                               C.c_uint32, C.c_int64, C.POINTER(PaOptions), C.POINTER(P)]
    L.pa_groupby_aggregate_chunked_keys.argtypes = [C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema), C.c_int32,
                                                    C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema), C.c_uint32, C.c_int64,
                                                    C.POINTER(PaOptions), C.POINTER(P)]
    L.pa_groupby_key_layout.argtypes = [P, C.POINTER(PaKeyLayout)]
    L.pa_key_layout_agree.argtypes = [C.POINTER(PaKeyLayout), C.c_int32, C.POINTER(PaKeyLayout)]
    L.pa_groupby_set_key_layout.argtypes = [P, C.POINTER(PaKeyLayout)]
    L.pa_merge_set_key_layout.argtypes = [P, C.POINTER(PaKeyLayout), C.POINTER(C.c_char_p)]
    L.pa_groupby_partials_export_padded.argtypes = [P, C.c_int32, P, C.c_int64]
    L.pa_merge_create_padded.argtypes = [P, C.c_int32, C.c_int64, C.c_uint32, C.c_char_p, C.c_char_p,
                                         C.POINTER(PaOptions), C.POINTER(P)]
    L.pa_comm_unique_id.argtypes = [P, C.c_int64]
    L.pa_comm_create.argtypes = [P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(P)]
    L.pa_comm_adopt.argtypes = [P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(P)]
    L.pa_comm_destroy.argtypes = [P]
    L.pa_comm_destroy.restype = None
    L.pa_groupby_sharded_aggregate.argtypes = [P, P, C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema), C.c_uint32, C.POINTER(P)]
    L.pa_comm_last_phases.argtypes = [P, C.POINTER(C.c_double)]
    L.pa_comm_last_exchange.argtypes = [P, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int64)]
    L.pa_comm_last_distinct.argtypes = [P, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.pa_comm_last_key_layout.argtypes = [P, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.pa_groupby_key_hash_seed.argtypes = [P, C.POINTER(C.c_uint64)]
    L.pa_groupby_set_key_hash_seed.argtypes = [P, C.c_uint64]
    L.pa_groupby_partials_count_utf8.argtypes = [P, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.pa_groupby_partials_export_utf8.argtypes = [P, C.c_int32, C.c_int32, P, C.c_int64, P, P, C.c_int64]
    L.pa_merge_key_strings.argtypes = [P, P, P, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_uint64), C.c_int32,
                                       C.POINTER(C.c_int32)]
    L.pa_comm_last_key_strings.argtypes = [P, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_uint64), C.POINTER(C.c_int32)]
    L.pa_synth_keys_i64.argtypes = [P, C.c_int64, C.c_int64, C.c_uint64, C.c_uint64, P]
    L.pa_synth_vals_f64.argtypes = [P, C.c_int64, C.c_int64, C.c_uint64, P]
    L.pa_synth_validity.argtypes = [P, C.c_int64, C.c_int64, C.c_uint64, C.c_uint32, P]
    L.pa_synth_timestamps.argtypes = [P, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_uint64, P]
    _lib = L
    return L
