/* pa_b200.h — C ABI of the B200-native group-by / resample hot path.
 *
 * This is the drop-in boundary for PandasArrow's group-by hash aggregation (SURVEY.md §8b).
 * The reference has no FFI of its own: its boundary is the C++ class surface
 *   pd::GroupBy            /root/reference/src/group_by.h:22-247
 *   pd::Resampler          /root/reference/src/group_by.h:255-299
 *   pd::resample           /root/reference/src/resample.h:51-122
 *   DataFrame::group_by / resample / downsample   /root/reference/src/dataframe.cpp:1227-1290
 * directly on top of arrow::compute.  The entry points below are what those classes bind to
 * instead of arrow::compute::Grouper / CallFunction; pandasarrow_b200/csrc/host/pd_groupby.h
 * is that binding (same class and method names as the reference), INTEGRATION.md shows the
 * patch a maintainer of the reference would apply.
 *
 * Data crosses the boundary as Arrow C Data Interface structs (arrow/c/abi.h): plain pointers
 * and sizes, no C++ or torch types.  Inputs are ArrowDeviceArray: device_type ARROW_DEVICE_CPU
 * buffers are copied host->device by the library, ARROW_DEVICE_CUDA buffers are used in place
 * (zero copy).  buffers[0] = validity bitmap (LSB first, may be NULL), buffers[1] = values;
 * `offset` and `null_count` are honoured.  Inputs are borrowed for the duration of the call that
 * receives them and until pa_groupby_destroy() for keys; the library never calls release() on an
 * input.  Outputs are host ArrowArray/ArrowSchema pairs owned by the caller (call release()).
 *
 * There is no CPU fallback: every call that computes fails with PA_ERR_CUDA when no CUDA device
 * is present.  All functions return 0 on success; pa_last_error() gives the thread-local message.
 */
#ifndef PA_B200_H
#define PA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- Arrow C Data Interface (verbatim ABI; guarded so arrow/c/abi.h may be included too) ---- */
#ifndef ARROW_C_DATA_INTERFACE
#define ARROW_C_DATA_INTERFACE
#define ARROW_FLAG_DICTIONARY_ORDERED 1
#define ARROW_FLAG_NULLABLE 2
#define ARROW_FLAG_MAP_KEYS_SORTED 4
struct ArrowSchema {
  const char* format;
  const char* name;
  const char* metadata;
  int64_t flags;
  int64_t n_children;
  struct ArrowSchema** children;
  struct ArrowSchema* dictionary;
  void (*release)(struct ArrowSchema*);
  void* private_data;
};
struct ArrowArray {
  int64_t length;
  int64_t null_count;
  int64_t offset;
  int64_t n_buffers;
  int64_t n_children;
  const void** buffers;
  struct ArrowArray** children;
  struct ArrowArray* dictionary;
  void (*release)(struct ArrowArray*);
  void* private_data;
};
#endif /* ARROW_C_DATA_INTERFACE */

#ifndef ARROW_C_DEVICE_DATA_INTERFACE
#define ARROW_C_DEVICE_DATA_INTERFACE
typedef int32_t ArrowDeviceType;
#define ARROW_DEVICE_CPU 1
#define ARROW_DEVICE_CUDA 2
#define ARROW_DEVICE_CUDA_HOST 3
struct ArrowDeviceArray {
  struct ArrowArray array;
  int64_t device_id;
  ArrowDeviceType device_type;
  void* sync_event;
  int64_t reserved[3];
};
#endif /* ARROW_C_DEVICE_DATA_INTERFACE */

/* ---- status codes ---- */
#define PA_OK 0
#define PA_ERR_INVALID 1     /* bad argument / unsupported type (message says which) */
#define PA_ERR_CUDA 2        /* CUDA runtime failure, or no device */
#define PA_ERR_NOT_IMPLEMENTED 3
#define PA_ERR_STATE 4       /* call order violated (e.g. fetch before aggregate) */

/* ---- aggregate selection: bit mask, outputs are produced in ascending bit order ----
 * Semantics follow the reference's per-group arrow::compute calls
 * (pd_core_macros.h:5-147, dataframe.cpp:1602-1806):
 *   SUM    int*->int64 (wraps), uint*->uint64, float/double->double; null for an all-null group
 *   MEAN   double (ints are accumulated in double); null for an all-null group
 *   COUNT  int64 number of non-null values
 *   MIN/MAX input dtype; NaN skipped unless the group is all-NaN; null for an all-null group
 *   FIRST/LAST value at the first/last row of the group, nulls NOT skipped (positional)
 * Second-stage aggregates (GROUPBY_AGG(product), GROUPBY_NUMERIC_AGG(variance|stddev), dataframe.cpp:1516-1536):
 * a second pass over keys + values after the fused one.  Row-range shards (multi-GPU, chunked) run it per shard and
 * merge the terms (PA_PARTIAL_WORDS_STAGE2 records): the per-shard M2 = sum of (x - mean_s)^2 combined with Chan's update
 * in source-rank order, the per-shard products multiplied in that order.  pa_groupby_aggregate on a merged handle
 * still refuses them.
 *   PRODUCT  int*->int64 (wraps), uint*->uint64, float/double->double; null for an all-null group
 *   VARIANCE/STDDEV  double, ddof 0, two-pass (mean, then squared deviations) as arrow::compute's
 *            scalar kernel; null for an all-null group (the reference's wrapper drops that validity)
 */
#define PA_AGG_SUM 1u
#define PA_AGG_MEAN 2u
#define PA_AGG_COUNT 4u
#define PA_AGG_MIN 8u
#define PA_AGG_MAX 16u
#define PA_AGG_FIRST 32u
#define PA_AGG_LAST 64u
#define PA_AGG_ALL 127u          /* everything the fused pass computes */
#define PA_AGG_PRODUCT 128u
#define PA_AGG_VARIANCE 256u
#define PA_AGG_STDDEV 512u
#define PA_AGG_STAGE2 896u       /* PRODUCT | VARIANCE | STDDEV */
#define PA_AGG_BOOL_ALL 1024u     /* GroupBy::all: boolean ('b') value columns only; bool result, null for an all-null group */
#define PA_AGG_BOOL_ANY 2048u     /* GroupBy::any */
#define PA_AGG_COUNT_DISTINCT 4096u /* GroupBy::count_distinct: int64 number of distinct non-null values (by bit pattern, as
                                      arrow's memo table: -0.0 and +0.0 are two values); < 2^31 rows per handle.  Across
                                      row-range shards through distinct-pair records (PA_DISTINCT_PAIR_WORDS) and
                                      pa_merge_distinct_pairs, or in one pa_groupby_sharded_aggregate step; not in
                                      pa_groupby_aggregate_chunked */

/* ---- kernel path selection (pa_options.path); AUTO is what a caller wants ---- */
#define PA_PATH_AUTO 0
#define PA_PATH_LOWCARD 1   /* shared-memory privatised tables only; fails if they overflow */
#define PA_PATH_GLOBAL 2    /* global-memory table with L2 atomics */

typedef struct pa_options {
  int32_t device;            /* CUDA device ordinal; -1 = current device */
  int32_t path;              /* PA_PATH_* */
  int64_t expected_groups;   /* hint for table sizing; 0 = unknown */
  void* cuda_stream;         /* cudaStream_t to run on; NULL = a stream owned by the handle */
  int64_t row_base;          /* global row number of local row 0 (multi-GPU row-range shards) */
  int64_t lowcard_no_dense;  /* 1 = the shared-memory path never uses dense (key - base) addressing, always hashes */
  int64_t no_partition;      /* 1 = never radix-partition the rows (bucketed path / table regions): plain global-table scan */
  int64_t bucket_bits;       /* tuning / tests: 0 = automatic; else level-1 bits | level-2 bits << 8 of the bucketed path */
  int64_t sm_reserve;        /* SMs the persistent shared-memory scan leaves free (0 = none): room for a concurrent NCCL
                                kernel / the merge of the previous multi-GPU step, whose CTAs cannot co-reside with a
                                scan CTA that owns ~200 KB of the SM's shared memory */
} pa_options;

typedef struct pa_groupby pa_groupby;      /* opaque: key columns + device group table */

const char* pa_last_error(void);
int pa_version(void);                       /* major*10000 + minor*100 + patch */
void pa_options_init(pa_options* opt);      /* fills defaults */
int pa_device_count(int* out);

/* pd::GroupBy::GroupBy / makeGroups (group_by.h:24-31, dataframe.cpp:1571-1600), stages 1-2.
 * keys[i] with key_schemas[i] describe the i-th key column (all the same length).  Supported key
 * formats: l L i I (int64/uint64/int32/uint32), ts* / tt* / td* (64-bit temporal), and
 * dictionary-encoded columns (the int32 indices are the key; the dictionary is not read).
 * Null keys form their own group.  A single key may also be utf8 / large_utf8 ("u" / "U": offsets + bytes, host or
 * device buffers, slices honoured).
 * A composite key (2 .. PA_MAX_KEY_COLS columns) that packs into 64 bits and has no utf8 column groups on its packed
 * word (see "composite keys across shards").  Any other composite key — wider than 64 bits, or with a utf8 / large_utf8
 * column — is a hashed key: a seeded 64-bit hash over all its columns in order (per column the null flag and, for a
 * valid slot, its value bits, a dictionary column's index, or a utf8 slot's length and bytes; never a null slot's
 * value) stands in for the key, 8 bytes per row computed here.  The first call that builds groups checks every row
 * against its group's first row (null flags, then the values of columns valid in both) and re-hashes with the next
 * seed on a mismatch, four seeds at most (then PA_ERR_STATE); until that check has passed, pa_groupby_aggregate_async
 * runs synchronously.  Group order and every result are those of the key columns themselves.  A hashed composite key
 * groups on one GPU: pa_groupby_key_layout / _set_key_layout, the partial-record and distinct-pair exports and
 * pa_groupby_sharded_aggregate return PA_ERR_NOT_IMPLEMENTED for it, and pa_groupby_aggregate_chunked_keys refuses
 * composite keys that do not pack, as it always has.
 * Work is lazy: the table is built by the first aggregate (fused with it) or by
 * pa_groupby_num_groups / pa_groupby_unique. */
int pa_groupby_create(const struct ArrowDeviceArray* keys, const struct ArrowSchema* key_schemas,
                      int32_t n_keys, const pa_options* opt, pa_groupby** out);

/* GroupBy::groupSize (group_by.h:33-36) */
int pa_groupby_num_groups(pa_groupby* g, int64_t* out);

/* GroupBy::unique (group_by.h:52-55): the key_i-th key column of the unique keys, in
 * first-appearance order, same type as the input key (dictionary keys: the int32 indices). */
int pa_groupby_unique(pa_groupby* g, int32_t key_i, struct ArrowArray* out, struct ArrowSchema* out_schema);

/* Stage 3, fused with stages 1-2: one pass over keys + values computing every aggregate in
 * agg_mask (GroupBy::sum/mean/count/min/max/first/last, pd_core_macros.h:5-147,
 * dataframe.cpp:1698-1806).  Value formats: g f l L i I s S c C (double, float, (u)int64/32/16/8),
 * 64-bit temporal types, and b (boolean: count / all / any only).  Results stay on the device until fetched. */
int pa_groupby_aggregate(pa_groupby* g, const struct ArrowDeviceArray* values,
                         const struct ArrowSchema* value_schema, uint32_t agg_mask);

/* Same, without waiting for the device when every input is device resident (ARROW_DEVICE_CUDA): the pass and
 * the result formatting are queued on the handle's stream and the call returns; the status words (group count,
 * overflow / fallback) are read by whichever call needs them next (fetch, num_groups, unique, last_timing,
 * sync, partials_count, the next aggregate ...), which also redoes the pass on the slower path if the
 * optimistic one did not apply.  The value buffers must stay alive until then.  Host inputs: identical to
 * pa_groupby_aggregate. */
int pa_groupby_aggregate_async(pa_groupby* g, const struct ArrowDeviceArray* values,
                               const struct ArrowSchema* value_schema, uint32_t agg_mask);

/* NDFrame<T>::sum / mean / min / max / count / first / last / min_max / agg
 * (/root/reference/src/ndframe.cpp:119,129,160-175,220,237-241): the whole column aggregated as ONE group by the
 * same fused pass (no key column is passed; a constant key is generated on the device).  Returns a handle with
 * num_groups <= 1 (0 for an empty column) whose results are read with pa_groupby_fetch.  skip_nulls != 0:
 * FIRST / LAST are the first / last VALID value, as arrow's scalar `first` / `last` kernels (GroupBy::first/last
 * stay positional); skip_nulls == 0: positional.  The caller applies arrow's "any null -> null" rule for
 * skip_nulls == 0 on sum / mean / min / max from the column's null_count. */
int pa_column_aggregate(const struct ArrowDeviceArray* values, const struct ArrowSchema* value_schema,
                        uint32_t agg_mask, int32_t skip_nulls, const pa_options* opt, pa_groupby** out);

/* Copies one finished aggregate (a single PA_AGG_* bit of the last aggregate call) to a host
 * Arrow array of length num_groups, first-appearance order. */
int pa_groupby_fetch(pa_groupby* g, uint32_t agg_bit, struct ArrowArray* out, struct ArrowSchema* out_schema);

/* Grouper::Consume equivalent (dataframe.cpp:1584): uint32 group id of every row, ids numbered in
 * first-appearance order.  Host array of length n_rows. */
int pa_groupby_row_ids(pa_groupby* g, struct ArrowArray* out, struct ArrowSchema* out_schema);

/* Grouper::MakeGroupings equivalent (dataframe.cpp:1586-1588): the row numbers of every group, group-contiguous
 * in result (first-appearance) order and ascending inside a group — the values (`rows`, int32[n_rows]) and the
 * offsets (int32[num_groups + 1]) of the ListArray<int32> the reference builds.  `rows` may be NULL (offsets only).
 * Built on the device on first use (row ids -> stable radix sort) and kept on the handle. */
int pa_groupby_groupings(pa_groupby* g, struct ArrowArray* offsets, struct ArrowSchema* offsets_schema,
                         struct ArrowArray* rows, struct ArrowSchema* rows_schema);

/* Grouper::ApplyGroupings equivalent for one column (dataframe.cpp:1546,1562): the column gathered on the device
 * into the order of pa_groupby_groupings — group j is the slice [offsets[j], offsets[j+1]).  Fixed-width columns
 * (1/2/4/8-byte elements), validity carried along.  Host array of the column's own type, n_rows long. */
int pa_groupby_take_grouped(pa_groupby* g, const struct ArrowDeviceArray* column, const struct ArrowSchema* schema,
                            struct ArrowArray* out, struct ArrowSchema* out_schema);

/* Device time (ms) of building the groupings, and of the last pa_groupby_take_grouped gather kernel. */
int pa_groupby_groupings_timing(pa_groupby* g, double* build_ms, double* take_ms);

/* Global row number (pa_options.row_base + local row) of the first row of every group, uint64, in
 * result order.  For merged handles: the minimum over all ranks. */
int pa_groupby_first_rows(pa_groupby* g, struct ArrowArray* out, struct ArrowSchema* out_schema);

/* Device time (ms, CUDA events on the handle's stream) of the last aggregate call: total and
 * per stage.  stage_ms[0]=key packing, [1]=scan kernel(s), [2]=merge/finalise, [3]=emit. */
int pa_groupby_last_timing(pa_groupby* g, double* total_ms, double stage_ms[4]);
/* Which path the last aggregate took (PA_PATH_LOWCARD / PA_PATH_GLOBAL) and how many of this
 * library's kernels it launched. */
int pa_groupby_last_path(pa_groupby* g, int32_t* path, int32_t* kernel_launches);
/* More about the last aggregate call: detail[0] = mode (0 n/a; shared-memory path: 1 dense key - base
 * addressing, 2 hash table; global path: 3 = shared-memory front table with spill,
 * 4 = rows radix-partitioned by table region first, detail[1] = log2(partitions); 5 = rows radix-partitioned into buckets that
 * are aggregated in shared memory, detail[1] = log2(buckets)), detail[1] = log2 of the accumulator replication (dense mode),
 * detail[2] = scan passes run (2 = a dense pass met a key outside its window and was rerun in hash
 * mode; +1 when the shared-memory tables overflowed and the global-table path ran), detail[3] = 0. */
int pa_groupby_last_detail(pa_groupby* g, int32_t detail[4]);
/* Blocks until everything queued on the handle's stream has finished. */
int pa_groupby_sync(pa_groupby* g);

void pa_groupby_destroy(pa_groupby* g);

/* pd::resample with a fixed-width rule (resample.h:91-122, resample.cpp:85-295): time-bucket
 * specialisation.  `index` is a sorted, null-free timestamp/int64 column; buckets are
 * [first + k*freq, first + (k+1)*freq) (closed_right: (..]) where `first` is anchored as
 * adjustDatesAnchored does (origin: 0 epoch, 1 start, 2 start_day, 3 end, 4 end_day, 5 custom).
 * Only non-empty buckets appear (the reference groups on per-row labels).  The returned handle
 * is a pa_groupby whose unique key is the bucket label: aggregate/fetch/unique work as above, on
 * a sorted-run segmented-reduction kernel instead of a hash table.  Throws-equivalents:
 * PA_ERR_INVALID for unsorted input, PA_ERR_NOT_IMPLEMENTED for up-sampling rules. */
int pa_resample_create(const struct ArrowDeviceArray* index, const struct ArrowSchema* index_schema,
                       int64_t freq_ns, int32_t closed_right, int32_t label_right, int32_t origin,
                       int64_t origin_custom_ns, int64_t offset_ns, const pa_options* opt,
                       pa_groupby** out);

/* pd::resample with a DateOffset rule (resample.cpp:248-267 makeGroupInfo's DateOffset branch, core.cpp:12-60
 * DateOffset::add, core.cpp:175-265 date_range, resample.cpp:180-200 adjustBinEdges).  offset_type is the reference's
 * DateOffset::Type (core.h:122-134); Day "D", WeekStart "WS", MonthStart "MS", QuarterStart "QS", YearStart "YS" are the
 * ones the reference's date_range accepts, the others return PA_ERR_NOT_IMPLEMENTED with the reference's message, as
 * does closed_right = 0 ("closed_left is not currently supported by DateOffset").  binner = date_range(first - freq,
 * last + freq, freq) at midnight; bucket i = (edge[i], edge[i+1]] with edge = binner + 1 day - 1 ns (edge = binner for
 * a plain "1D" rule), labelled binner[i] (label_right: binner[i+1]).  The index must be a sorted, null-free
 * timestamp[ns] column.  Same handle semantics as pa_resample_create. */
#define PA_OFFSET_DAY 0
#define PA_OFFSET_MONTH_END 1
#define PA_OFFSET_QUARTER_START 2
#define PA_OFFSET_QUARTER_END 3
#define PA_OFFSET_WEEK_START 4
#define PA_OFFSET_WEEK_END 5
#define PA_OFFSET_MONTH_START 6
#define PA_OFFSET_YEAR_END 7
#define PA_OFFSET_YEAR_START 8
int pa_resample_create_calendar(const struct ArrowDeviceArray* index, const struct ArrowSchema* index_schema,
                                int32_t offset_type, int32_t multiplier, int32_t closed_right, int32_t label_right,
                                const pa_options* opt, pa_groupby** out);

/* DataFrame::downsample (dataframe.cpp:1265-1290): groups on the per-row label
 * arrow::compute::FloorTemporal / CeilTemporal(index, RoundTemporalOptions(multiple, unit, week_starts_monday,
 * ceil_is_strictly_greater = false, calendar_based_origin)) — computed on the device, bit-identical to arrow's
 * kernels without a time zone — minus one day for W / M / Q / Y, exactly as the reference does.  `unit` is the
 * reference's rule letter: N U L S T H D W M Q Y.  `index` is a timestamp column (any resolution for the fixed
 * units, [ns] for W / M / Q / Y; may be unsorted; null timestamps form the null-key group).  The returned handle is
 * an ordinary pa_groupby whose unique key is the label column. */
int pa_downsample_create(const struct ArrowDeviceArray* index, const struct ArrowSchema* index_schema, int32_t multiple,
                         char unit, int32_t closed_label_right, int32_t week_starts_monday, int32_t calendar_based_origin,
                         const pa_options* opt, pa_groupby** out);

/* ---- ingest (SURVEY.md §8f rank 4): DataFrame::readBinary / readParquet (dataframe.cpp:757-791, 646-683) leave host
 * Arrow arrays (an IPC blob, a decoded Parquet table).  pa_column_to_device copies one such array to the device ONCE —
 * pageable memory through the library's pinned, multi-threaded staging pipeline, i.e. at the PCIe rate — and returns an
 * ArrowDeviceArray with device_type ARROW_DEVICE_CUDA that owns its device buffers (out->array.release frees them;
 * `schema` keeps describing it).  Every other entry point then uses the column in place: the constructor and every
 * aggregate after it stop paying PCIe.  Fixed-width, boolean and (large_)utf8 columns; slices are honoured. */
int pa_column_to_device(const struct ArrowDeviceArray* host, const struct ArrowSchema* schema, const pa_options* opt,
                        struct ArrowDeviceArray* out);

/* ---- stable argsort (SURVEY.md §8f rank 4): Series::argsort / Series::sort / DataFrame::sort_index / sort_values
 * (series.cpp:864-868,978-992, dataframe.cpp:1062-1071,1188-1208), which the reference gets from arrow::compute
 * "array_sort_indices" + Take.  Same ordering rules: stable, NaNs after every number and nulls after the NaNs in BOTH
 * orders.  Numeric and 64-bit temporal columns, < 2^31 rows.  The returned handle is a pa_groupby in "sorted" state:
 * pa_sort_indices returns the uint64 indices, pa_groupby_take_grouped(handle, column) returns any column of the same
 * length in sorted order (scatter-shaped take, fixed-width and boolean columns), pa_groupby_destroy frees it. */
int pa_sort_create(const struct ArrowDeviceArray* values, const struct ArrowSchema* schema, int32_t ascending,
                   const pa_options* opt, pa_groupby** out);
int pa_sort_indices(pa_groupby* sorted, struct ArrowArray* out, struct ArrowSchema* out_schema);

/* ---- multi-GPU: row-range shards, hash-partitioned partial aggregates, merge (SURVEY.md §8e) ----
 * The reference has no multi-device path.  Each rank aggregates its shard (pa_options.row_base =
 * global row number of its first row), buckets its groups by owner = hash(key) % n_parts into
 * fixed-size records, exchanges them with an all-to-all (NCCL over NVLink; the caller owns the
 * communicator — see pandasarrow_b200/distributed.py), and merges what it received.  A record is
 * PA_PARTIAL_WORDS 64-bit words. */
#define PA_PARTIAL_WORDS 11
/* Number of this handle's groups owned by each of n_parts ranks (host array, after an aggregate). */
int pa_groupby_partials_count(pa_groupby* g, int32_t n_parts, int64_t* counts_host);
/* Writes the records, grouped by owner rank in ascending order, into caller-provided DEVICE memory
 * (capacity_records >= sum of counts).  Must follow pa_groupby_partials_count with the same n_parts.
 * Always PA_PARTIAL_WORDS-word records, also after an aggregate with product / variance / stddev. */
int pa_groupby_partials_export(pa_groupby* g, int32_t n_parts, void* dev_records, int64_t capacity_records);
/* Stage-2 records: the PA_PARTIAL_WORDS words, then this handle's M2 = sum of (x - mean)^2 of the group (double bits;
 * mean = sum / count as the second pass computed it) and its product (raw 64 bits: double, or wrapped (u)int64).  Same
 * preconditions as pa_groupby_partials_export; PA_ERR_STATE when the last aggregate computed none of
 * product / variance / stddev (a flag in the record says which of the two terms it holds). */
#define PA_PARTIAL_WORDS_STAGE2 13
int pa_groupby_partials_export_stage2(pa_groupby* g, int32_t n_parts, void* dev_records, int64_t capacity_records);
/* Joins received records (DEVICE memory, grouped by source rank; counts_by_source on the host) by key,
 * folds them in source-rank order and orders the groups by global first row.  The returned handle
 * answers num_groups / unique / fetch for the aggregates in agg_mask (PA_AGG_ALL, PA_AGG_STAGE2, and with value_format
 * "b" PA_AGG_BOOL_ALL / PA_AGG_BOOL_ANY bits: those merge the records' min / max and count).  The
 * records are PA_PARTIAL_WORDS_STAGE2 words wide exactly when agg_mask has a PA_AGG_STAGE2 bit (then PA_ERR_STATE if
 * a record lacks the terms asked for), PA_PARTIAL_WORDS otherwise.  value_format / key_format are
 * the Arrow format strings of the value and (single) key column; a composite key travels as its packed word: pass "L" and
 * then pa_merge_set_key_layout.  PA_AGG_COUNT_DISTINCT is not a record aggregate:
 * see pa_merge_distinct_pairs. */
int pa_merge_create(const void* dev_records, const int64_t* counts_by_source, int32_t n_sources, uint32_t agg_mask,
                    const char* value_format, const char* key_format, const pa_options* opt, pa_groupby** out);

/* count_distinct across shards.  A per-group count does not merge (a value may occur on several shards), so every shard
 * ships its distinct (key, value) pairs to the key's owner, which deduplicates across sources.  A distinct-pair record is
 * PA_DISTINCT_PAIR_WORDS 64-bit words: [0] the key, [1] the value widened to 64 bits exactly as count_distinct compares
 * it (-0.0 / +0.0 and NaNs with different payloads stay distinct), [2] flags, bit 0 = null key.  A handle whose last
 * aggregate computed count_distinct keeps its D distinct pairs (12 bytes each; at most half of what that aggregate's
 * sort needs) until the next aggregate or pa_groupby_destroy. */
#define PA_DISTINCT_PAIR_WORDS 3
/* Number of this handle's distinct pairs owned by each of n_parts ranks (1 <= n_parts <= 64), routed like the group
 * records (the null key goes to rank 0).  PA_ERR_STATE when the last aggregate did not compute count_distinct or the
 * handle is merged.  Pairs of a utf8 key carry its hash: merge them after pa_merge_key_strings. */
int pa_groupby_distinct_pairs_count(pa_groupby* g, int32_t n_parts, int64_t* counts_host);
/* Writes the pairs, grouped by owner rank in ascending order, into caller-provided DEVICE memory (capacity_pairs >= sum of
 * counts).  Must follow pa_groupby_distinct_pairs_count with the same n_parts. */
int pa_groupby_distinct_pairs_export(pa_groupby* g, int32_t n_parts, void* dev_pairs, int64_t capacity_pairs);
/* Adds a PA_AGG_COUNT_DISTINCT output (int64, the merged handle's group order, 0 for a group without pairs) to a handle
 * made by pa_merge_create or pa_groupby_sharded_aggregate, from the received pairs (DEVICE memory, grouped by source;
 * counts_by_source on the host; at most 2^32 - 2 in all).  A second call replaces the first.  The count is exact and
 * does not depend on the order of arrival.  The owner-side set takes 32 bytes per received pair while the call runs.
 * PA_ERR_STATE on a handle that is not merged, and when a pair names a key that no merged record carried (an
 * inconsistent exchange). */
int pa_merge_distinct_pairs(pa_groupby* merged, const void* dev_pairs, const int64_t* counts_by_source, int32_t n_sources);

/* Low-latency variant for few groups — no host round trip before the collective.  Writes, for every
 * destination rank, a fixed-size block of (1 + block_records) records into caller-provided DEVICE memory
 * (n_parts blocks): record 0 is a header (word 0 = number of records that follow, or all-ones when this
 * handle has more than block_records groups), then the records that rank owns.  The call is stream ordered
 * (no synchronisation).  All ranks exchange the blocks with an equal-split all-to-all and hand what they
 * received (n_sources blocks, in source-rank order) to pa_merge_create_padded, which returns
 * PA_ERR_STATE when any source sent the overflow marker (every rank sees it: fall back to
 * pa_groupby_partials_count / _export / pa_merge_create).  PA_AGG_ALL bits only (PA_PARTIAL_WORDS-word records). */
int pa_groupby_partials_export_padded(pa_groupby* g, int32_t n_parts, void* dev_blocks, int64_t block_records);
int pa_merge_create_padded(const void* dev_blocks, int32_t n_sources, int64_t block_records, uint32_t agg_mask,
                           const char* value_format, const char* key_format, const pa_options* opt, pa_groupby** out);

/* ---- utf8 / large_utf8 keys across shards ----
 * A single utf8 key is grouped by a seeded 64-bit hash of its bytes, and its records carry that hash as their key word.
 * Two things make the records alone unsafe across shards: a handle whose own byte check found two strings under one
 * hash re-hashes with the next seed (so shards may hash one string differently), and two strings of different shards
 * may share a hash (which no shard can see).  So every record travels with its group's key bytes, all shards hash with
 * one seed, and the owner compares the bytes of every record of a merged group with those of its representative (the
 * record carrying the group's global first row: the first string in row order).  The plain pa_groupby_partials_count /
 * _export / _export_stage2 / _export_padded and pa_merge_create_padded refuse utf8 keys.
 *
 * The hash seed of a handle with a hashed key — one utf8 / large_utf8 key, or a composite key that does not pack into
 * 64 bits (pa_groupby_create) — 0 at creation, raised by the handle's own check on a collision; PA_ERR_INVALID for any
 * other handle.  Test hook: with the environment variable PA_TEST_STR_HASH_BITS=b, hashes made under seed 0 keep only
 * their low b bits (utf8 keys and hashed composite keys alike), so that different keys share a hash on demand. */
int pa_groupby_key_hash_seed(pa_groupby* g, uint64_t* seed);
/* Re-hashes the key column with `seed` (the largest seed of all shards, see pa_merge_key_strings).  Completes a pending
 * aggregate first; groups, outputs, groupings, distinct pairs and stage-2 terms are dropped like pa_groupby_set_key_layout
 * does, and the next aggregate checks the grouping byte for byte again (which may raise the seed once more).  Equal to
 * the current seed: no-op.  PA_ERR_INVALID for a handle that is not a single utf8 key. */
int pa_groupby_set_key_hash_seed(pa_groupby* g, uint64_t seed);
/* Records (as pa_groupby_partials_count) and key bytes owned by each of n_parts ranks, after an aggregate. */
int pa_groupby_partials_count_utf8(pa_groupby* g, int32_t n_parts, int64_t* records_host, int64_t* bytes_host);
/* Writes the records (PA_PARTIAL_WORDS words, or PA_PARTIAL_WORDS_STAGE2 when stage2 != 0, as
 * pa_groupby_partials_export / _export_stage2), one uint32 key length per record (0 for the null key) and the key
 * bytes, all grouped by owner rank in the same order, into caller-provided DEVICE memory (capacity_records >= the
 * records, capacity_bytes >= the key bytes of pa_groupby_partials_count_utf8, which must come first with the same
 * n_parts).  Record i's bytes follow those of records 0 .. i-1. */
int pa_groupby_partials_export_utf8(pa_groupby* g, int32_t n_parts, int32_t stage2, void* dev_records, int64_t capacity_records,
                                    void* dev_lengths, void* dev_bytes, int64_t capacity_bytes);
/* Owner side, on a handle made by pa_merge_create with key_format "u" / "U" from utf8 records (whose record buffer must
 * still be alive): attaches the merged groups' key strings from the received lengths and bytes (DEVICE memory, grouped
 * by source like the records; records_by_source as given to pa_merge_create, bytes_by_source and every source's hash
 * seed on the host).  Every record's bytes are compared with its group's representative's; when two different strings
 * share a merged group, *collided = 1, no strings are attached, and the caller's ranks agree a retry with the next seed
 * (4 seeds at most).  Otherwise *collided = 0 and pa_groupby_unique(merged, 0) returns utf8 (key_format "u") or
 * large_utf8 ("U"); before that it returns PA_ERR_STATE, and so does pa_merge_distinct_pairs.  The merged handle keeps
 * only its G representative strings.  PA_ERR_INVALID when the seeds differ: hashes of one string under two seeds are
 * two groups, which nothing after the merge can detect. */
int pa_merge_key_strings(pa_groupby* merged, const void* dev_lengths, const void* dev_bytes, const int64_t* records_by_source,
                         const int64_t* bytes_by_source, const uint64_t* seed_by_source, int32_t n_sources, int32_t* collided);

/* ---- composite keys across shards ----
 * A composite key is packed into one 64-bit word per row: column j takes bits[j] value bits, then one null bit when
 * nullable[j], columns in order from bit 0.  Records, owner routing and the merge treat that word as the key.  A handle
 * packs with the layout its own data implies: a column carries a null bit only when the column handed to
 * pa_groupby_create has a validity bitmap and a nonzero null_count, and a dictionary column takes bits_for(dictionary
 * length) bits.  Shards of one frame can therefore pack the same group into different words.  Before their records
 * meet, all shards agree on one layout (pa_key_layout_agree over every shard's pa_groupby_key_layout) and repack to it
 * (pa_groupby_set_key_layout); pa_groupby_sharded_aggregate does both by itself.  A composite key that does not pack
 * (a hashed composite key, pa_groupby_create) has no layout: these calls, the partial-record and distinct-pair exports
 * and the sharded step return PA_ERR_NOT_IMPLEMENTED for it.  Whether a shard's key packs depends on its own nulls and
 * dictionaries, so in the sharded step a hashed rank still takes part in the layout gather (with an empty layout) and
 * every rank fails together. */
#define PA_MAX_KEY_COLS 4
typedef struct pa_key_layout {
  int32_t n_keys;                               /* 2 .. PA_MAX_KEY_COLS */
  int32_t width[PA_MAX_KEY_COLS];               /* bytes of the key column: 4 or 8 */
  int32_t bits[PA_MAX_KEY_COLS];                /* value bits (dictionary: bits for its length) */
  int32_t nullable[PA_MAX_KEY_COLS];            /* 0 / 1: the field carries a null bit */
  uint64_t dict_fingerprint[PA_MAX_KEY_COLS];   /* 64-bit hash of the dictionary's values; 0 = not a dictionary */
} pa_key_layout;
/* The current layout of a composite (2+ column) key handle.  The dictionary fingerprints hash each dictionary's format,
 * then every entry's validity and bytes; they are computed on the first call and kept (a dictionary on the device is
 * copied to the host for that).  PA_ERR_INVALID for a single-key, resample or merged handle. */
int pa_groupby_key_layout(pa_groupby* g, pa_key_layout* out);
/* The layout every shard packs with, from all n shards' layouts.  Column count, widths, bits and dictionary
 * fingerprints must be equal on every input (otherwise PA_ERR_INVALID naming the column; for dictionaries: encode the
 * column against one dictionary shared by all shards); a column is nullable when it is nullable on any input.
 * PA_ERR_NOT_IMPLEMENTED when the result needs more than 64 bits.  Every shard that applies this to the same inputs
 * gets the same answer, so all fail together before any record moves. */
int pa_key_layout_agree(const pa_key_layout* all, int32_t n, pa_key_layout* out);
/* Repacks a composite key handle's keys under `layout`, which must dominate its own (same column count, widths, bits
 * and fingerprints; nullable wherever its own is), else PA_ERR_INVALID.  Completes a pending aggregate first; the
 * groups, outputs, groupings, distinct pairs and stage-2 terms of earlier aggregates are dropped (the next call
 * recomputes them; group order and values do not change).  Equal to the current layout: no-op. */
int pa_groupby_set_key_layout(pa_groupby* g, const pa_key_layout* layout);
/* Gives a merged handle (pa_merge_create / pa_merge_create_padded with key_format "L", the packed word) the composite
 * key: pa_groupby_unique(merged, j) then returns column j with format key_formats[j] (a dictionary column: its index
 * format), null where the null bit is set.  Does not complete a pending padded merge. */
int pa_merge_set_key_layout(pa_groupby* merged, const pa_key_layout* layout, const char* const* key_formats);

/* Host frames larger than free device memory (or than 2^32-2 rows): the columns are aggregated chunk_rows rows at a
 * time — each chunk copied through the pinned staging pipeline, aggregated with row_base = its first row and exported as
 * partial records — and the chunks' records are merged like ranks' (sources folded in row order, groups in global
 * first-appearance order).  Single key column; sum / mean / count / min / max / first / last / product / variance / stddev
 * (those three travel in PA_PARTIAL_WORDS_STAGE2-word records) and all / any of boolean columns; not count_distinct.
 * A utf8 / large_utf8 key: every chunk hashes with one seed and exports its key bytes next to its records; a chunk
 * whose own check raises the seed, or a merge that finds two strings under one hash, redoes the chunks with the next
 * seed (4 at most).
 * `merged_out` answers
 * num_groups / unique / fetch like a merged multi-GPU handle.  At most 64 chunks.
 * pa_groupby_aggregate_chunked is pa_groupby_aggregate_chunked_keys with n_keys = 1. */
int pa_groupby_aggregate_chunked(const struct ArrowDeviceArray* keys, const struct ArrowSchema* key_schema,
                                 const struct ArrowDeviceArray* values, const struct ArrowSchema* value_schema,
                                 uint32_t agg_mask, int64_t chunk_rows, const pa_options* opt, pa_groupby** merged_out);
/* The same with n_keys key columns (a composite key as pa_groupby_create takes it).  Chunks are views of the same
 * columns, so every chunk packs with the layout of the whole columns; the merged handle carries that layout and
 * answers pa_groupby_unique for every key column.  A composite key must pack into 64 bits and hold no utf8 column
 * (dictionary-encode it): decided from the whole columns before any chunk, PA_ERR_NOT_IMPLEMENTED otherwise. */
int pa_groupby_aggregate_chunked_keys(const struct ArrowDeviceArray* keys, const struct ArrowSchema* key_schemas, int32_t n_keys,
                                      const struct ArrowDeviceArray* values, const struct ArrowSchema* value_schema,
                                      uint32_t agg_mask, int64_t chunk_rows, const pa_options* opt, pa_groupby** merged_out);

/* ---- the same exchange driven from C: communicator handle + one call per step (SURVEY.md §8b, §8e).
 * pa_comm wraps an NCCL communicator over the GPUs of one node (NVLink / NVSwitch).  Rank 0 obtains an id with
 * pa_comm_unique_id (PA_COMM_ID_BYTES bytes), every rank receives it by any out-of-band channel (MPI, a file,
 * torch.distributed ...) and calls pa_comm_create; or an existing ncclComm_t is adopted (not destroyed by
 * pa_comm_destroy).  pa_groupby_sharded_aggregate then runs, on the handle's stream: the local fused pass over this
 * rank's row shard (pa_options.row_base = its first global row), the owner bucketing, the exchange of counts
 * (ncclAllGather) and records (grouped ncclSend / ncclRecv), and the owner-side merge; `merged_out` answers
 * num_groups / unique / fetch / first_rows for the groups with hash(key) % world == rank.  Send / receive / merge
 * scratch stays on the communicator between steps.  Aggregates: PA_AGG_ALL and PA_AGG_STAGE2 bits (the latter travel in
 * PA_PARTIAL_WORDS_STAGE2-word records, see pa_groupby_partials_export_stage2), PA_AGG_BOOL_ALL / PA_AGG_BOOL_ANY
 * (boolean columns), and PA_AGG_COUNT_DISTINCT: the pairs are counted per owner before the count gather, which carries
 * both counts, travel in a second grouped send / receive after the records and are deduplicated on the merged handle
 * (pa_merge_distinct_pairs); pair send / receive / set scratch stays on the communicator too.  A composite key handle
 * starts every step with one more ncclAllGather, of every rank's pa_key_layout, agrees on a layout
 * (pa_key_layout_agree; all ranks fail together when the layouts do not agree), repacks when it differs from the
 * handle's own (pa_groupby_set_key_layout) and hands the merged handle that layout and its key formats.  A utf8 key
 * handle adds its hash seed and its key bytes per owner to the count gather; when the seeds differ every rank re-hashes
 * with the largest and redoes the step.  The key lengths and bytes follow the records in one more grouped send /
 * receive, the owner checks them (pa_merge_key_strings), and one ncclAllReduce (max) of the collision word follows;
 * after a collision every rank redoes the step with the next seed.  Four seeds at most, then PA_ERR_STATE on every rank.
 * Other single-key and resample steps issue no extra collective. */
#define PA_COMM_ID_BYTES 128
typedef struct pa_comm pa_comm;
int pa_comm_unique_id(void* out_id, int64_t capacity_bytes);
int pa_comm_create(const void* id, int32_t world, int32_t rank, int32_t device, pa_comm** out);
int pa_comm_adopt(void* nccl_comm, int32_t world, int32_t rank, int32_t device, pa_comm** out);
void pa_comm_destroy(pa_comm* c);
int pa_groupby_sharded_aggregate(pa_groupby* g, pa_comm* c, const struct ArrowDeviceArray* values,
                                 const struct ArrowSchema* value_schema, uint32_t agg_mask, pa_groupby** merged_out);
/* Device time (ms) of the last step's phases: [0] local pass, [1] count + export, [2] exchange, [3] merge, [4] total. */
int pa_comm_last_phases(pa_comm* c, double phase_ms[5]);
/* How the last step's partial aggregates travelled: bytes per group record (32: compact records of sum / mean of floats /
 * count; 88: the full PA_PARTIAL_WORDS record; 104: the PA_PARTIAL_WORDS_STAGE2 record), whether the local pass handed over the bucketed path's unordered group
 * records without ordering them first (0 / 1), and the slots of the merge's join table. */
int pa_comm_last_exchange(pa_comm* c, int32_t* record_bytes, int32_t* unordered_export, int64_t* merge_table_slots);
/* The last step's count_distinct exchange: distinct pairs this rank sent and received, and the slots of its owner-side
 * set (all 0 when the step computed no count_distinct). */
int pa_comm_last_distinct(pa_comm* c, int64_t* pairs_sent, int64_t* pairs_received, int64_t* set_slots);
/* The last step's composite-key agreement, outside the phases above: device time (ms) of the layout gather (copy in,
 * ncclAllGather, copy out) and of the repack (0 when the handle already packed with the agreed layout); both 0 for a
 * single-key or resample step. */
int pa_comm_last_key_layout(pa_comm* c, double* agree_ms, double* repack_ms);
/* The last step's utf8 key exchange: key bytes this rank sent and received, the seed all ranks hashed with, and the
 * number of attempts the step took (1 without a seed change); all 0 for a step without a utf8 key. */
int pa_comm_last_key_strings(pa_comm* c, int64_t* bytes_sent, int64_t* bytes_received, uint64_t* seed, int32_t* attempts);

/* ---- synthetic workload generator (SURVEY.md §8d), used by bench.py and the tests so that the
 * same counter-based splitmix64 streams exist on host and device without PCIe staging.
 * All pointers are DEVICE pointers; `first_row` offsets the counter (row-range shards). ---- */
int pa_synth_keys_i64(void* dev_out, int64_t n, int64_t first_row, uint64_t n_groups, uint64_t seed, void* cuda_stream);
int pa_synth_vals_f64(void* dev_out, int64_t n, int64_t first_row, uint64_t seed, void* cuda_stream);
int pa_synth_validity(void* dev_bitmap_out, int64_t n, int64_t first_row, uint64_t seed, uint32_t null_every, void* cuda_stream);
int pa_synth_timestamps(void* dev_out, int64_t n, int64_t first_row, int64_t t0_ns, int64_t step_ns, uint64_t seed, void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* PA_B200_H */
