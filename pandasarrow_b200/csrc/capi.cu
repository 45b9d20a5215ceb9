// C ABI of the B200 group-by path (include/pa_b200.h).  Host-side orchestration only: column
// marshalling from the Arrow C Data Interface, path selection, kernel launches, result export.
// No computation happens on the host and there is no CPU fallback.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cuda_runtime.h>
#include <nccl.h>

#include <algorithm>
#include <cstdarg>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/pa_b200.h"
#include "emit.cuh"
#include "gtable.cuh"
#include "lowcard.cuh"
#include "lowcard_known.cuh"
#include "merge.cuh"
#include "partition.cuh"
#include "bucketed.cuh"
#include "resample.cuh"
#include "rowids.cuh"
#include "stage2.cuh"
#include "groupings.cuh"
#include "distinct.cuh"
#include "temporal.cuh"
#include "order.cuh"
#include "csort.cuh"
#include "sort.cuh"
#include "strkeys.cuh"
#include "rowkeys.cuh"

using namespace pa;

namespace {

thread_local std::string g_err;

int set_err(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CUDA_TRY(expr)                                                                             \
  do {                                                                                             \
    cudaError_t e__ = (expr);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      return set_err(PA_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

#define PA_TRY(expr)        \
  do {                      \
    int rc__ = (expr);      \
    if (rc__ != PA_OK) return rc__; \
  } while (0)

// Stream-ordered device allocation; the pool keeps freed memory so that repeated aggregate
// calls (bench steps) do not pay cudaMalloc.
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  cudaStream_t s = nullptr;
  bool plain = false;     // cudaMalloc / cudaFree instead of the stream-ordered pool: for buffers that outlive the streams they are used on
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept { *this = std::move(o); }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) { reset(); p = o.p; bytes = o.bytes; s = o.s; plain = o.plain; o.p = nullptr; o.bytes = 0; }
    return *this;
  }
  ~DevBuf() { reset(); }
  void reset() {
    if (p) { if (plain) cudaFree(p); else cudaFreeAsync(p, s); }
    p = nullptr;
    bytes = 0;
  }
  int alloc(size_t n, cudaStream_t stream) {
    if (n == 0) n = 16;
    if (plain) {
      if (p && bytes >= n) return PA_OK;
      reset();
      CUDA_TRY(cudaMalloc(&p, n));
      bytes = n;
      return PA_OK;
    }
    if (p && s == stream && bytes >= n) return PA_OK;   // recycled handle: the old block is big enough
    reset();
    s = stream;
    static const bool dbg = getenv("PA_DEBUG_ALLOC") != nullptr;
    const auto t0 = std::chrono::steady_clock::now();
    CUDA_TRY(cudaMallocAsync(&p, n, stream));
    if (dbg) {
      const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
      if (ms > 2.0) fprintf(stderr, "[pa alloc] %.1f MB took %.1f ms\n", n / 1048576.0, ms);
    }
    bytes = n;
    return PA_OK;
  }
  template <typename T>
  T* as() const { return static_cast<T*>(p); }
};

struct Column {
  const void* data = nullptr;       // device pointer, already advanced by `offset` elements
  const uint8_t* valid = nullptr;   // device validity bitmap (not advanced) or null
  int64_t bit_off = 0;
  int64_t n = 0;
  int width = 0;                    // bytes per element
  int vc = VC_I;                    // value class (value columns)
  std::string format;               // Arrow format string of the (index) type
  bool is_dict = false;
  bool is_bool = false;             // Arrow boolean (bit-packed) unpacked to one byte per value in own_data
  int64_t dict_len = 0;
  // dictionary key column: the (borrowed) dictionary and its fingerprint (dict_fingerprint), computed on first need
  const ArrowArray* dict = nullptr;
  const ArrowSchema* dict_schema = nullptr;
  bool dict_on_dev = false;
  uint64_t dict_fp = 0;
  DevBuf own_data, own_valid;       // set when the input lived on the host (or was unpacked)
  DevBuf own_bits;                  // boolean host input: the packed bits on the device
  // utf8 / large_utf8 KEY columns (strkeys.cuh): the key word is a hash (pa_groupby::hashed), the strings stay reachable here
  bool is_str = false;
  StrCol str{};
  DevBuf own_offsets, own_bytes;
};

int parse_format(const char* f, int* width, int* vc) {
  if (!f) return set_err(PA_ERR_INVALID, "schema has no format string");
  switch (f[0]) {
    case 'g': *width = 8; *vc = VC_F; return PA_OK;
    case 'f': *width = 4; *vc = VC_F; return PA_OK;
    case 'l': *width = 8; *vc = VC_I; return PA_OK;
    case 'L': *width = 8; *vc = VC_U; return PA_OK;
    case 'i': *width = 4; *vc = VC_I; return PA_OK;
    case 'I': *width = 4; *vc = VC_U; return PA_OK;
    case 's': *width = 2; *vc = VC_I; return PA_OK;
    case 'S': *width = 2; *vc = VC_U; return PA_OK;
    case 'c': *width = 1; *vc = VC_I; return PA_OK;
    case 'C': *width = 1; *vc = VC_U; return PA_OK;
    case 'b': *width = 1; *vc = VC_U; return PA_OK;   // boolean: unpacked to bytes by load_column
    case 't':
      // tss/tsm/tsu/tsn timestamps, tD* durations, ttu/ttn time64, tdm date64: 64-bit; tdD date32, tts/ttm: 32-bit
      if (f[1] == 's' || f[1] == 'D') { *width = 8; *vc = VC_I; return PA_OK; }
      if (f[1] == 't') { *width = (f[2] == 'u' || f[2] == 'n') ? 8 : 4; *vc = VC_I; return PA_OK; }
      if (f[1] == 'd') { *width = (f[2] == 'm') ? 8 : 4; *vc = VC_I; return PA_OK; }
      break;
    default: break;
  }
  return set_err(PA_ERR_INVALID, "unsupported Arrow format '%s' (fixed-width numeric / temporal only)", f);
}

// Host -> device copy of a column buffer.  Pinned source: one cudaMemcpyAsync at the PCIe rate.  Pageable source
// (ordinary Arrow heap buffers — what pd::DataFrame holds —, an IPC blob, Parquet-decoded columns): the driver would
// bounce it through its own small staging area at a fraction of that rate, so anything large goes through the
// library's two pinned staging buffers, filled by a few host threads while the previous chunk is on the wire.
namespace {
constexpr size_t H2D_CHUNK = 8u << 20;            // bytes per staging buffer (two per worker); PA_H2D_CHUNK_MB overrides
constexpr size_t H2D_STAGED_MIN = 16u << 20;      // smaller copies are not worth the pipeline
constexpr int H2D_MAX_WORKERS = 16;
constexpr int H2D_MAX_BUFS = 4;
struct H2dWorker {
  void* pin[H2D_MAX_BUFS] = {};
  cudaEvent_t done[H2D_MAX_BUFS] = {};
  cudaEvent_t fin = nullptr;
  cudaStream_t stream = nullptr;
};
struct H2dStage {
  std::mutex mu;
  H2dWorker w[H2D_MAX_WORKERS];
  cudaEvent_t start = nullptr;
  bool ok = false, tried = false;
  int workers = 1;
  size_t chunk = H2D_CHUNK;
  int bufs = 2;                                    // staging buffers per worker; PA_H2D_BUFS overrides
};
H2dStage g_h2d_dev[16];   // one per device: streams and events belong to a device

bool h2d_stage_ready(H2dStage& g) {
  if (g.tried) return g.ok;
  g.tried = true;
  if (const char* e = getenv("PA_H2D_STAGED")) { if (atoi(e) == 0) return false; }
  const unsigned hc = std::thread::hardware_concurrency();
  g.workers = static_cast<int>(std::max(1u, std::min(8u, hc ? hc / 2 : 4u)));
  if (const char* e = getenv("PA_H2D_THREADS")) g.workers = std::max(1, std::min(H2D_MAX_WORKERS, atoi(e)));
  if (const char* e = getenv("PA_H2D_BUFS")) g.bufs = std::max(2, std::min(H2D_MAX_BUFS, atoi(e)));
  if (const char* e = getenv("PA_H2D_CHUNK_MB")) g.chunk = static_cast<size_t>(std::max(1, std::min(64, atoi(e)))) << 20;
  if (cudaEventCreateWithFlags(&g.start, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return false; }
  for (int i = 0; i < g.workers; ++i) {
    H2dWorker& w = g.w[i];
    bool good = cudaStreamCreateWithFlags(&w.stream, cudaStreamNonBlocking) == cudaSuccess &&
                cudaEventCreateWithFlags(&w.fin, cudaEventDisableTiming) == cudaSuccess;
    for (int b = 0; b < g.bufs && good; ++b)
      good = cudaHostAlloc(&w.pin[b], g.chunk, cudaHostAllocPortable) == cudaSuccess &&
             cudaEventCreateWithFlags(&w.done[b], cudaEventDisableTiming) == cudaSuccess;
    if (!good) { cudaGetLastError(); return false; }
  }
  g.ok = true;
  return true;
}
}  // namespace

// Every worker thread owns a contiguous slice of the copy, two pinned buffers and a stream: it copies a chunk into
// one buffer while the DMA engine drains the other.  The destination was allocated in stream order on `st`, so the
// worker streams start behind an event on `st`, and `st` continues behind the workers' last copies.
int h2d_copy(void* dst, const void* src, size_t bytes, cudaStream_t st) {
  if (!bytes) return PA_OK;
  bool pageable = false;
  if (bytes >= H2D_STAGED_MIN) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, src) != cudaSuccess) { cudaGetLastError(); pageable = true; }
    else pageable = at.type == cudaMemoryTypeUnregistered;
  }
  if (!pageable) {
    CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
    return PA_OK;
  }
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  H2dStage& g = g_h2d_dev[dev & 15];
  std::lock_guard<std::mutex> lock(g.mu);
  if (!h2d_stage_ready(g)) {
    CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
    return PA_OK;
  }
  CUDA_TRY(cudaEventRecord(g.start, st));
  const int T = g.workers;
  const size_t per = ((bytes + T - 1) / T + 4095) & ~static_cast<size_t>(4095);
  std::vector<cudaError_t> err(T, cudaSuccess);
  auto work = [&](int t) {
    H2dWorker& w = g.w[t];
    cudaError_t e = cudaSetDevice(dev);
    const size_t lo = per * t, hi = std::min(bytes, lo + per);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(w.stream, g.start, 0);
    int b = 0;
    for (size_t off = lo; off < hi && e == cudaSuccess; off += g.chunk, b = b + 1 == g.bufs ? 0 : b + 1) {
      const size_t len = std::min(g.chunk, hi - off);
      e = cudaEventSynchronize(w.done[b]);                 // the previous copy out of this buffer has finished
      if (e != cudaSuccess) break;
      memcpy(w.pin[b], static_cast<const char*>(src) + off, len);
      e = cudaMemcpyAsync(static_cast<char*>(dst) + off, w.pin[b], len, cudaMemcpyHostToDevice, w.stream);
      if (e == cudaSuccess) e = cudaEventRecord(w.done[b], w.stream);
    }
    if (e == cudaSuccess) e = cudaEventRecord(w.fin, w.stream);
    err[t] = e;
  };
  std::vector<std::thread> pool;
  for (int t = 1; t < T; ++t) pool.emplace_back(work, t);
  work(0);
  for (auto& th : pool) th.join();
  for (int t = 0; t < T; ++t) {
    if (err[t] != cudaSuccess) return set_err(PA_ERR_CUDA, "staged host-to-device copy failed: %s", cudaGetErrorString(err[t]));
    CUDA_TRY(cudaStreamWaitEvent(st, g.w[t].fin, 0));
  }
  return PA_OK;
}

// Bring one primitive Arrow array onto the device (or borrow it when it already is there).
int load_column(const ArrowDeviceArray* da, const ArrowSchema* sc, cudaStream_t st, int device, Column* out) {
  const ArrowArray& a = da->array;
  if (a.n_buffers < 2) return set_err(PA_ERR_INVALID, "expected a primitive array with 2 buffers, got %lld", (long long)a.n_buffers);
  PA_TRY(parse_format(sc->format, &out->width, &out->vc));
  out->format = sc->format;
  out->is_dict = sc->dictionary != nullptr;
  out->dict_len = (a.dictionary != nullptr) ? a.dictionary->length : 0;
  out->dict = a.dictionary;
  out->dict_schema = sc->dictionary;
  out->dict_on_dev = da->device_type == ARROW_DEVICE_CUDA;
  out->n = a.length;
  const bool has_nulls = a.null_count != 0 && a.buffers[0] != nullptr;
  const char* values = static_cast<const char*>(a.buffers[1]);
  out->is_bool = sc->format[0] == 'b';
  if (out->is_bool) {
    // Bit-packed values -> one byte per value on the device (the kernels then see a uint8 column of 0 / 1).
    if (da->device_type == ARROW_DEVICE_CUDA && da->device_id != device)
      return set_err(PA_ERR_INVALID, "array lives on device %lld, handle on %d", (long long)da->device_id, device);
    const bool on_dev = da->device_type == ARROW_DEVICE_CUDA;
    if (!on_dev && da->device_type != ARROW_DEVICE_CPU && da->device_type != ARROW_DEVICE_CUDA_HOST)
      return set_err(PA_ERR_INVALID, "unsupported device_type %d", (int)da->device_type);
    if (on_dev && da->sync_event) CUDA_TRY(cudaStreamWaitEvent(st, *static_cast<cudaEvent_t*>(da->sync_event), 0));
    const int64_t first_byte = a.offset / 8;
    const size_t nbytes = static_cast<size_t>((a.offset + a.length + 7) / 8 - first_byte);
    const uint8_t* bits = reinterpret_cast<const uint8_t*>(values) + first_byte;
    if (!on_dev) {
      PA_TRY(out->own_bits.alloc(std::max<size_t>(nbytes, 1), st));
      PA_TRY(h2d_copy(out->own_bits.p, bits, nbytes, st));
      bits = out->own_bits.as<uint8_t>();
    }
    PA_TRY(out->own_data.alloc(static_cast<size_t>(std::max<int64_t>(a.length, 1)), st));
    if (a.length > 0) {
      const int grid = static_cast<int>(std::min<int64_t>((a.length + 255) / 256, 148 * 16));
      k_unpack_bool<<<grid, 256, 0, st>>>(bits, a.offset % 8, a.length, out->own_data.as<uint8_t>());
      CUDA_TRY(cudaGetLastError());
    }
    out->data = out->own_data.p;
    if (has_nulls) {
      if (on_dev) {
        out->valid = static_cast<const uint8_t*>(a.buffers[0]);
        out->bit_off = a.offset;
      } else {
        PA_TRY(out->own_valid.alloc(nbytes, st));
        PA_TRY(h2d_copy(out->own_valid.p, static_cast<const uint8_t*>(a.buffers[0]) + first_byte, nbytes, st));
        out->valid = out->own_valid.as<uint8_t>();
        out->bit_off = a.offset % 8;
      }
    }
    return PA_OK;
  }
  if (da->device_type == ARROW_DEVICE_CUDA) {
    if (da->device_id != device) return set_err(PA_ERR_INVALID, "array lives on device %lld, handle on %d", (long long)da->device_id, device);
    out->data = values ? values + a.offset * out->width : nullptr;
    out->valid = has_nulls ? static_cast<const uint8_t*>(a.buffers[0]) : nullptr;
    out->bit_off = a.offset;
    if (da->sync_event) CUDA_TRY(cudaStreamWaitEvent(st, *static_cast<cudaEvent_t*>(da->sync_event), 0));
  } else if (da->device_type == ARROW_DEVICE_CPU || da->device_type == ARROW_DEVICE_CUDA_HOST) {
    const size_t bytes = static_cast<size_t>(a.length) * out->width;
    PA_TRY(out->own_data.alloc(bytes, st));
    PA_TRY(h2d_copy(out->own_data.p, values + a.offset * out->width, bytes, st));
    out->data = out->own_data.p;
    if (has_nulls) {
      // copy the bytes that cover bits [offset, offset+length); keep the sub-byte offset
      const int64_t first_byte = a.offset / 8;
      const size_t nbytes = static_cast<size_t>((a.offset + a.length + 7) / 8 - first_byte);
      PA_TRY(out->own_valid.alloc(nbytes, st));
      PA_TRY(h2d_copy(out->own_valid.p, static_cast<const uint8_t*>(a.buffers[0]) + first_byte, nbytes, st));
      out->valid = out->own_valid.as<uint8_t>();
      out->bit_off = a.offset % 8;
    }
  } else {
    return set_err(PA_ERR_INVALID, "unsupported device_type %d", (int)da->device_type);
  }
  return PA_OK;
}

// utf8 / large_utf8 key column: offsets + bytes onto the device (or borrowed); setup_keys hashes the key.
int load_string_key(const ArrowDeviceArray* da, const ArrowSchema* sc, cudaStream_t st, int device, Column* out) {
  const ArrowArray& a = da->array;
  if (a.n_buffers < 3) return set_err(PA_ERR_INVALID, "utf8 array needs 3 buffers (validity, offsets, data), got %lld", (long long)a.n_buffers);
  const bool wide = sc->format[0] == 'U';
  const int ow = wide ? 8 : 4;
  out->format = sc->format;
  out->is_str = true;
  out->width = 8;
  out->vc = VC_U;
  out->n = a.length;
  const bool has_nulls = a.null_count != 0 && a.buffers[0] != nullptr;
  const char* offs = static_cast<const char*>(a.buffers[1]) + a.offset * ow;
  const uint8_t* bytes = static_cast<const uint8_t*>(a.buffers[2]);
  if (da->device_type == ARROW_DEVICE_CUDA) {
    if (da->device_id != device) return set_err(PA_ERR_INVALID, "array lives on device %lld, handle on %d", (long long)da->device_id, device);
    if (da->sync_event) CUDA_TRY(cudaStreamWaitEvent(st, *static_cast<cudaEvent_t*>(da->sync_event), 0));
    out->str.offsets = offs;
    out->str.bytes = bytes;
    out->valid = has_nulls ? static_cast<const uint8_t*>(a.buffers[0]) : nullptr;
    out->bit_off = a.offset;
  } else if (da->device_type == ARROW_DEVICE_CPU || da->device_type == ARROW_DEVICE_CUDA_HOST) {
    const int64_t n = a.length;
    int64_t first = 0, last = 0;
    if (a.buffers[1]) {
      first = wide ? reinterpret_cast<const int64_t*>(offs)[0] : reinterpret_cast<const int32_t*>(offs)[0];
      last = wide ? reinterpret_cast<const int64_t*>(offs)[n] : reinterpret_cast<const int32_t*>(offs)[n];
    }
    PA_TRY(out->own_offsets.alloc(static_cast<size_t>(n + 1) * ow, st));
    if (a.buffers[1]) PA_TRY(h2d_copy(out->own_offsets.p, offs, static_cast<size_t>(n + 1) * ow, st));
    else CUDA_TRY(cudaMemsetAsync(out->own_offsets.p, 0, static_cast<size_t>(n + 1) * ow, st));
    PA_TRY(out->own_bytes.alloc(static_cast<size_t>(std::max<int64_t>(last - first, 1)), st));
    if (last > first) PA_TRY(h2d_copy(out->own_bytes.p, bytes + first, static_cast<size_t>(last - first), st));
    out->str.offsets = out->own_offsets.p;
    out->str.bytes = out->own_bytes.as<uint8_t>() - first;       // offsets stay absolute
    if (has_nulls) {
      const int64_t first_byte = a.offset / 8;
      const size_t nbytes = static_cast<size_t>((a.offset + a.length + 7) / 8 - first_byte);
      PA_TRY(out->own_valid.alloc(nbytes, st));
      PA_TRY(h2d_copy(out->own_valid.p, static_cast<const uint8_t*>(a.buffers[0]) + first_byte, nbytes, st));
      out->valid = out->own_valid.as<uint8_t>();
      out->bit_off = a.offset % 8;
    }
  } else {
    return set_err(PA_ERR_INVALID, "unsupported device_type %d", (int)da->device_type);
  }
  out->str.wide = wide ? 1 : 0;
  return PA_OK;
}

struct KeyField {
  int width = 8, bits = 64, shift = 0, nullable = 0;
};

struct AggOut {
  uint32_t bit = 0;
  std::string format;
  int width = 8;
  bool nullable = true;
  DevBuf values, valid;
};

}  // namespace

struct pa_groupby {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int num_sms = 148;
  pa_options opt{};
  int64_t n = 0;
  // keys
  std::vector<Column> keys;
  std::vector<KeyField> fields;
  bool packed = false;
  // hashed key — one utf8 column, or a composite key that does not pack into 64 bits: the key word is a seeded 64-bit
  // hash (strkeys.cuh, rowkeys.cuh) in packed_keys; key_verified once a pass has checked every row against its group's
  // first row, key_seed counts the re-hashes after a collision
  bool hashed = false;
  bool key_verified = false;
  uint64_t key_seed = 0;
  DevBuf packed_keys;
  const void* key_data = nullptr;   // what the scan kernels read
  const uint8_t* key_valid = nullptr;
  int64_t key_bit_off = 0;
  int key_width = 8;
  // resample mode (time-bucket specialisation)
  bool resample = false;
  std::string index_format;
  ResampleSpec rs{};
  DevBuf rs_edges, rs_labels;             // calendar rules: bucket edges / labels on the device (rs.edges / rs.labels)
  // group table in first-appearance order
  bool have_groups = false;
  // Sharded step with compact records: the bucketed path may leave its unordered per-bucket group records (BkRec32) as
  // the result of the local pass — the merge orders by GLOBAL first row anyway — instead of ranking and gathering them
  // into the GroupResult (8.5 ms per 100 M groups).  want_unordered: asked for by pa_groupby_sharded_aggregate;
  // unordered: this pass did so (g->G records at unordered_recs; the GroupResult and the outputs were NOT touched).
  bool want_unordered = false, unordered = false;
  const void* unordered_recs = nullptr;
  uint32_t unordered_G = 0;
  uint32_t G = 0;
  uint32_t res_cap = 0;
  DevBuf r_key, r_kind, r_sum, r_dsum, r_count, r_first, r_last, r_min, r_max;
  GroupResult res{};
  // outputs of the last aggregate
  std::vector<AggOut> outs;
  // product / variance / stddev of the last aggregate: which of them it computed (PA_AGG_STAGE2 bits, 0 = none) and its
  // per-group terms — M2 = sum of (x - mean)^2 and the product — kept until the next aggregate for the stage-2 partial
  // export (pa_groupby_partials_export_stage2); on a merged handle, the merged terms
  uint32_t s2_ext = 0;
  DevBuf s2_m2, s2_prod;
  // count_distinct of the last aggregate: its distinct (local group id, value bits) pairs, cd_n of them, kept until the
  // next aggregate for pa_groupby_distinct_pairs_export (12 bytes per pair)
  bool cd_have = false;
  uint64_t cd_n = 0;
  DevBuf cd_id, cd_bits;
  int dp_parts_n = 0;                     // pa_groupby_distinct_pairs_count: n_parts and the pairs per owner
  std::vector<int64_t> dp_counts;
  bool last_wide = false;
  int last_vc = VC_I, last_vw = 8;
  std::string last_vfmt = "l";
  // multi-GPU
  int parts_n = 0;
  std::vector<int64_t> parts_counts;
  std::vector<int64_t> ks_counts;         // utf8 key: key bytes per owner (pa_groupby_partials_count_utf8)
  bool merged = false;
  // merged handle of a utf8 key (key format "u" / "U"): its G representative strings once pa_merge_key_strings has
  // attached them — int64 offsets, bytes, and rows 0 .. G-1 for unique_strings
  bool ks_str = false, ks_have = false;
  DevBuf ks_off, ks_bytes, ks_rows;
  const void* ks_recs = nullptr;          // pa_merge_create's records (the caller's buffer), ks_nrec of ks_words words
  int ks_words = 0;
  uint64_t ks_nrec = 0;
  DevBuf m_count64, m_first_val, m_last_val, m_first_valid, m_last_valid, m_first_row_g;
  // bookkeeping
  DevBuf status;
  int last_path = 0, last_launches = 0;
  int last_mode = 0, last_rlog = 0, last_passes = 0;
  const uint32_t* emit_G_dev = nullptr;   // run_emit: exact group count lives on the device (g->G is an upper bound)
  bool poolable = false;                  // merged handle built by the fused small merge: recycled on destroy
  // deferred (asynchronous) aggregate: kernels are queued, the status words have not been read yet
  bool pending = false;
  Column pending_val;                     // borrowed device pointers of the value column (no ownership)
  bool pending_has_val = false;
  uint32_t pending_mask = 0;
  uint32_t pending_prev_G = 0;
  bool pending_had_groups = false;
  bool pending_lk_record = false;         // the pending pass records the dense facts below
  // Dense low-cardinality facts of this handle's keys (lowcard_known.cuh): window, group count, id -> rank, count /
  // first row / key by rank.  Recorded by a full dense narrow-set pass; trusted (lk_valid) once the host has read that
  // pass's clean status; dropped with everything else computed from the key words and on any aborted pass.
  DevBuf lk_buf;
  bool lk_valid = false;
  // deferred fused merge of padded blocks (multi-GPU): status not read yet; the caller keeps the blocks alive
  bool pending_merge = false;
  const void* pm_blocks = nullptr;
  int32_t pm_nsrc = 0;
  int64_t pm_block_records = 0;
  uint32_t pm_mask = 0;
  std::string pm_vfmt, pm_kfmt;
  float last_total_ms = 0;
  float stage_ms[4] = {0, 0, 0, 0};
  cudaEvent_t ev[10] = {};                // [6..7]: groupings build, [8..9]: last grouped take
  // group materialisation (groupings.cuh), built on first use; keys are immutable so it never goes stale
  DevBuf grp_order, grp_offsets, grp_dest;
  bool have_groupings = false;
  bool sorted_state = false;              // handle made by pa_sort_create: grp_order / grp_dest hold the sorted row order
  // Scratch of the global-table / resample passes, kept between calls on the handle: returning multi-GB blocks to
  // the stream-ordered pool and asking for them again fragments it (cudaMallocAsync then takes 50-1700 ms per call
  // at 100 M groups); a repeated aggregate on the same handle reuses these without touching the allocator.
  struct Scratch {
    DevBuf table, p_keys, p_vals, p_rows, p_counts, krange, c_first, c_slot, s_first, s_slot, cub_tmp, bnd, bitmap, prefix8, tile_sums;
    // bucketed path (bucketed.cuh): second-level rows, histograms / cursors, sketch, unordered groups
    DevBuf q_keys, q_vals, q_rows, rp_fine, rp_counts1, rp_counts2, rp_ends1, rp_ends2, rp_tiles, rp_hll, rp_next, u_rec, u_first;
  } scr;
  double est_groups = 0;                  // bucketed path: HyperLogLog estimate of the group count
  bool bk_have_hist = false;              // bucketed path: level-1 fine histogram + sketch of this handle's keys exist
  int bk_bits = -1, bk_b1 = -1;           // bucketed path: plan whose offsets / bucket ends are cached in scr.rp_*
};

namespace {

int alloc_result(pa_groupby* g, uint32_t cap, bool wide, bool need_dsum) {
  cudaStream_t st = g->stream;
  if (cap == 0) cap = 1;
  g->res_cap = cap;
  PA_TRY(g->r_key.alloc(sizeof(uint64_t) * cap, st));
  PA_TRY(g->r_kind.alloc(cap, st));
  PA_TRY(g->r_sum.alloc(sizeof(uint64_t) * cap, st));
  PA_TRY(g->r_count.alloc(sizeof(uint32_t) * cap, st));
  PA_TRY(g->r_first.alloc(sizeof(uint32_t) * cap, st));
  PA_TRY(g->r_last.alloc(sizeof(uint32_t) * cap, st));
  g->res = GroupResult{};
  g->res.key = g->r_key.as<uint64_t>();
  g->res.key_kind = g->r_kind.as<uint8_t>();
  g->res.sum = g->r_sum.as<uint64_t>();
  g->res.count = g->r_count.as<uint32_t>();
  g->res.first_row = g->r_first.as<uint32_t>();
  g->res.last_row = g->r_last.as<uint32_t>();
  if (wide) {
    PA_TRY(g->r_min.alloc(sizeof(uint64_t) * cap, st));
    PA_TRY(g->r_max.alloc(sizeof(uint64_t) * cap, st));
    g->res.min_ord = g->r_min.as<uint64_t>();
    g->res.max_ord = g->r_max.as<uint64_t>();
    if (need_dsum) {
      PA_TRY(g->r_dsum.alloc(sizeof(double) * cap, st));
      g->res.dsum = g->r_dsum.as<double>();
    }
  }
  return PA_OK;
}

int run_resample(pa_groupby* g, const Column* val, uint32_t mask, bool wide);

bool is_wide(uint32_t mask, int vc) {
  return (mask & (AGG_MIN | AGG_MAX | AGG_LAST)) || ((mask & AGG_MEAN) && vc != VC_F);
}

// ------------------------------ low-cardinality path ------------------------------
enum LcOutcome { LC_DONE = 0, LC_DENSE_MISS = 1, LC_OVERFLOW = 2 };

bool lc_is_wide(uint32_t mask, int vc) { return is_wide(mask, vc); }

template <int VC, bool WIDE>
int launch_lowcard_t(pa_groupby* g, const LcArgs& a, const LmArgs& m, int grid, bool fast, bool hash_kernel) {
  using Cfg = LcCfg<VC, WIDE>;
  cudaStream_t st = g->stream;
  k_lowcard_prep<<<LC_PREP_GRID, 256, 0, st>>>(a);
  CUDA_TRY(cudaGetLastError());
  if (hash_kernel) {
    using L = LcSmem<VC, WIDE, true>;
    auto scan = fast ? k_lowcard_scan<VC, WIDE, true, false> : k_lowcard_scan<VC, WIDE, false, false>;
    CUDA_TRY(cudaFuncSetAttribute(scan, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(L::TOTAL)));
    scan<<<grid, L::WARPS * 32, L::TOTAL, st>>>(a);
  } else {
    using L = LcSmem<VC, WIDE, false>;
    auto scan = fast ? k_lowcard_scan<VC, WIDE, true, true> : k_lowcard_scan<VC, WIDE, false, true>;
    CUDA_TRY(cudaFuncSetAttribute(scan, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(L::TOTAL)));
    scan<<<grid, L::WARPS * 32, L::TOTAL, st>>>(a);
  }
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaEventRecord(g->ev[2], st));
  k_lowcard_merge<VC, WIDE><<<(Cfg::GP + 7) / 8, 256, 0, st>>>(m);
  CUDA_TRY(cudaGetLastError());
  k_lowcard_rank<VC, WIDE><<<(Cfg::GP + LR_THREADS / 32 - 1) / (LR_THREADS / 32), LR_THREADS, 0, st>>>(m);
  CUDA_TRY(cudaGetLastError());
  g->last_launches += 4;
  return PA_OK;
}

// one persistent CTA per SM the handle may use (the order of the floating-point sums depends on it)
int lc_grid(const pa_groupby* g) {
  return std::max<int>(1, g->num_sms - static_cast<int>(std::max<int64_t>(0, std::min<int64_t>(g->opt.sm_reserve, g->num_sms - 1))));
}

// The handle's fact buffers (lowcard_known.cuh): LkHead | id_rank [GP] | count [GP] | first [GP] | key [GP] | kind [GP]
int lk_facts(pa_groupby* g, LkFacts* f) {
  constexpr size_t gp = LcCfg<VC_F, false>::GP;
  PA_TRY(g->lk_buf.alloc(sizeof(LkHead) + gp * (4 + 4 + 4 + 8 + 1), g->stream));
  char* p = g->lk_buf.as<char>();
  f->head = reinterpret_cast<LkHead*>(p);
  f->key = reinterpret_cast<uint64_t*>(p + sizeof(LkHead));
  f->id_rank = reinterpret_cast<uint32_t*>(f->key + gp);
  f->count = f->id_rank + gp;
  f->first = f->count + gp;
  f->kind = reinterpret_cast<uint8_t*>(f->first + gp);
  return PA_OK;
}

int run_lowcard(pa_groupby* g, const Column* val, uint32_t mask, bool wide, bool force_hash, LcOutcome* outcome,
                bool deferred = false) {
  cudaStream_t st = g->stream;
  const int grid = lc_grid(g);
  const int vc = val ? val->vc : VC_I;
  const bool kwide = lc_is_wide(mask, vc);
  // a dense pass of the narrow set over a value column without a bitmap (count = group size) records the facts of
  // the handle's keys for the sum-only passes after it
  const bool record = !g->lk_valid && !kwide && !force_hash && val && !val->valid;
  const bool dsum = kwide && vc != VC_F;
  const int gp = lc_gmax(vc, kwide) + 2;
  const size_t np = static_cast<size_t>(grid) * gp;
  DevBuf p_sum, p_dsum, p_count, p_first, p_last, p_min, p_max, merged, dir;
  PA_TRY(p_sum.alloc(np * 8, st));
  PA_TRY(p_count.alloc(np * 4, st));
  PA_TRY(p_first.alloc(np * 4, st));
  if (kwide) {
    PA_TRY(p_last.alloc(np * 4, st));
    PA_TRY(p_min.alloc(np * 8, st));
    PA_TRY(p_max.alloc(np * 8, st));
    if (dsum) PA_TRY(p_dsum.alloc(np * 8, st));
  }
  // merged-by-id scratch: sum, dsum, min, max (8 B each) then count, first, last (4 B each)
  const size_t gp8 = static_cast<size_t>(gp) * 8, gp4 = static_cast<size_t>(gp) * 4;
  PA_TRY(merged.alloc(gp8 * 4 + gp4 * 3, st));
  // directory: LcPrep | key_by_id | gt_keys | gt_ids
  const size_t dir_bytes = sizeof(LcPrep) + static_cast<size_t>(LC_GMAX_MAX) * 8 + static_cast<size_t>(LC_GT_CAP) * 12;
  PA_TRY(dir.alloc(dir_bytes, st));
  CUDA_TRY(cudaMemsetAsync(dir.p, 0, sizeof(LcPrep), st));
  CUDA_TRY(cudaMemsetAsync(g->status.p, 0, sizeof(uint32_t) * ST_WORDS, st));
  PA_TRY(alloc_result(g, gp, wide, vc != VC_F));

  LcArgs a{};
  a.keys = g->key_data;
  a.kvalid = g->key_valid;
  a.koff = g->key_bit_off;
  a.kw = g->key_width;
  a.vals = val ? val->data : nullptr;
  a.vvalid = val ? val->valid : nullptr;
  a.voff = val ? val->bit_off : 0;
  a.vw = val ? val->width : 8;
  a.n = g->n;
  a.force_hash = force_hash ? 1 : 0;
  a.hash_rlog = 0;
  if (force_hash) {
    // replicas per id for few scattered keys, from a group count this handle already knows (its keys never change) or
    // the caller's hint; a count that turns out too small overflows to the global path like any other overflow
    const uint64_t known = g->have_groups ? g->G : static_cast<uint64_t>(std::max<int64_t>(g->opt.expected_groups, 0));
    const uint64_t cap = static_cast<uint64_t>(lc_gmax_hash(vc, kwide));
    if (known > 0) while (a.hash_rlog < 5 && ((known + 1) << (a.hash_rlog + 1)) <= cap) ++a.hash_rlog;
  }
  a.agg_mask = mask;
  char* d = dir.as<char>();
  a.dir.prep = reinterpret_cast<LcPrep*>(d);
  a.dir.key_by_id = reinterpret_cast<unsigned long long*>(d + sizeof(LcPrep));
  a.dir.gt_keys = a.dir.key_by_id + LC_GMAX_MAX;
  a.dir.gt_ids = reinterpret_cast<unsigned int*>(a.dir.gt_keys + LC_GT_CAP);
  a.p_sum = p_sum.as<uint64_t>();
  a.p_dsum = p_dsum.as<double>();
  a.p_count = p_count.as<uint32_t>();
  a.p_first = p_first.as<uint32_t>();
  a.p_last = p_last.as<uint32_t>();
  a.p_min = p_min.as<uint64_t>();
  a.p_max = p_max.as<uint64_t>();
  a.status = g->status.as<uint32_t>();
  const bool aligned = (reinterpret_cast<uintptr_t>(a.keys) % 8 == 0) && (reinterpret_cast<uintptr_t>(a.vals) % 8 == 0);
  const bool fast = a.vals && aligned && a.kw == 8 && a.vw == 8 && !a.kvalid && !a.vvalid;
  LmArgs m{};
  m.part = a;
  m.grid = grid;
  m.gp = gp;
  char* mp = merged.as<char>();
  m.m_sum = reinterpret_cast<uint64_t*>(mp);
  m.m_dsum = reinterpret_cast<double*>(mp + gp8);
  m.m_min = reinterpret_cast<uint64_t*>(mp + gp8 * 2);
  m.m_max = reinterpret_cast<uint64_t*>(mp + gp8 * 3);
  m.m_count = reinterpret_cast<uint32_t*>(mp + gp8 * 4);
  m.m_first = m.m_count + gp;
  m.m_last = m.m_first + gp;
  m.out = g->res;
  m.status = a.status;
  CUDA_TRY(cudaEventRecord(g->ev[1], st));
  if (kwide) {
    if (vc == VC_F) PA_TRY((launch_lowcard_t<VC_F, true>(g, a, m, grid, fast, force_hash)));
    else if (vc == VC_I) PA_TRY((launch_lowcard_t<VC_I, true>(g, a, m, grid, fast, force_hash)));
    else PA_TRY((launch_lowcard_t<VC_U, true>(g, a, m, grid, fast, force_hash)));
  } else {
    if (vc == VC_F) PA_TRY((launch_lowcard_t<VC_F, false>(g, a, m, grid, fast, force_hash)));
    else if (vc == VC_I) PA_TRY((launch_lowcard_t<VC_I, false>(g, a, m, grid, fast, force_hash)));
    else PA_TRY((launch_lowcard_t<VC_U, false>(g, a, m, grid, fast, force_hash)));
  }
  if (record) {
    LkFacts f;
    PA_TRY(lk_facts(g, &f));
    k_lowcard_known_record<<<1, LK_REC_THREADS, 0, st>>>(m, f);
    CUDA_TRY(cudaGetLastError());
    g->last_launches += 1;
  }
  CUDA_TRY(cudaEventRecord(g->ev[3], st));
  if (deferred) {   // the scratch buffers above are released in stream order; the status is read by finish_pending()
    g->G = static_cast<uint32_t>(gp);   // upper bound until then
    g->pending_lk_record = record;
    *outcome = LC_DONE;
    return PA_OK;
  }
  uint32_t h_status[ST_WORDS];
  CUDA_TRY(cudaMemcpyAsync(h_status, g->status.p, sizeof h_status, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  if (h_status[ST_OVERFLOW]) *outcome = LC_OVERFLOW;
  else if (h_status[ST_DENSE_MISS]) *outcome = LC_DENSE_MISS;
  else { *outcome = LC_DONE; g->G = h_status[ST_NGROUPS]; }
  if (*outcome != LC_DONE) g->lk_valid = false;
  else if (record && h_status[ST_MODE] == 1u) g->lk_valid = true;
  g->last_mode = static_cast<int>(h_status[ST_MODE]);
  g->last_rlog = static_cast<int>(h_status[ST_RLOG]);
  if (h_status[ST_DENSE_MISS] != 2u) g->last_passes += 1;   // (2 = the dense kernel declined before scanning a row)
  return PA_OK;
}

// Sum-only pass of a handle whose dense facts are valid (lowcard_known.cuh): narrow set, value column without a bitmap.
bool lk_applies(const pa_groupby* g, const Column* val, uint32_t mask) {
  if (!g->lk_valid || !val || val->valid || lc_is_wide(mask, val->vc)) return false;
  const char* e = std::getenv("PA_LC_NO_KNOWN");   // (read per call: A/B runs in one process)
  return !(e && std::atoi(e) != 0);
}

template <int VC>
int launch_lowcard_known_t(pa_groupby* g, const LcArgs& a, const LmArgs& m, int grid, bool fast, const LkFacts& f) {
  cudaStream_t st = g->stream;
  auto scan = fast ? k_lowcard_sums<VC, true> : k_lowcard_sums<VC, false>;
  CUDA_TRY(cudaFuncSetAttribute(scan, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(LkSmem::TOTAL)));
  scan<<<grid, LkSmem::WARPS * 32, LkSmem::TOTAL, st>>>(a, f.head);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaEventRecord(g->ev[2], st));
  k_lowcard_sums_merge<VC><<<(LcCfg<VC, false>::GP + 7) / 8, 256, 0, st>>>(m, f);
  CUDA_TRY(cudaGetLastError());
  g->last_launches += 2;
  return PA_OK;
}

int run_lowcard_known(pa_groupby* g, const Column* val, uint32_t mask, LcOutcome* outcome, bool deferred) {
  cudaStream_t st = g->stream;
  const int grid = lc_grid(g);
  const int vc = val->vc;
  const int gp = lc_gmax(vc, false) + 2;
  const size_t np = static_cast<size_t>(grid) * gp;
  DevBuf p_sum, p_seen;
  PA_TRY(p_sum.alloc(np * 8, st));
  PA_TRY(p_seen.alloc(np * 4, st));
  CUDA_TRY(cudaMemsetAsync(g->status.p, 0, sizeof(uint32_t) * ST_WORDS, st));
  PA_TRY(alloc_result(g, gp, false, vc != VC_F));
  LkFacts f;
  PA_TRY(lk_facts(g, &f));

  LcArgs a{};
  a.keys = g->key_data;
  a.kvalid = g->key_valid;
  a.koff = g->key_bit_off;
  a.kw = g->key_width;
  a.vals = val->data;
  a.vw = val->width;
  a.n = g->n;
  a.agg_mask = mask;
  a.p_sum = p_sum.as<uint64_t>();
  a.p_count = p_seen.as<uint32_t>();   // 1 where the CTA met the id
  a.status = g->status.as<uint32_t>();
  const bool aligned = (reinterpret_cast<uintptr_t>(a.keys) % 8 == 0) && (reinterpret_cast<uintptr_t>(a.vals) % 8 == 0);
  const bool fast = a.vals && aligned && a.kw == 8 && a.vw == 8 && !a.kvalid;
  LmArgs m{};
  m.part = a;
  m.grid = grid;
  m.gp = gp;
  m.out = g->res;
  m.status = a.status;
  CUDA_TRY(cudaEventRecord(g->ev[1], st));
  if (vc == VC_F) PA_TRY(launch_lowcard_known_t<VC_F>(g, a, m, grid, fast, f));
  else if (vc == VC_I) PA_TRY(launch_lowcard_known_t<VC_I>(g, a, m, grid, fast, f));
  else PA_TRY(launch_lowcard_known_t<VC_U>(g, a, m, grid, fast, f));
  CUDA_TRY(cudaEventRecord(g->ev[3], st));
  g->pending_lk_record = false;
  *outcome = LC_DONE;
  if (deferred) {
    g->G = static_cast<uint32_t>(gp);   // upper bound until finish_pending()
    return PA_OK;
  }
  uint32_t h_status[ST_WORDS];
  CUDA_TRY(cudaMemcpyAsync(h_status, g->status.p, sizeof h_status, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  if (h_status[ST_ABORT]) {   // a key outside the recorded window, or a group the facts do not have
    g->lk_valid = false;
    *outcome = LC_DENSE_MISS;
  } else {
    g->G = h_status[ST_NGROUPS];
  }
  g->last_mode = static_cast<int>(h_status[ST_MODE]);
  g->last_rlog = static_cast<int>(h_status[ST_RLOG]);
  g->last_passes += 1;
  return PA_OK;
}

// Orders G compacted (first_row, slot) pairs by first row WITHOUT a sort (order.cuh): rank query on a bitmap of the
// first rows.  Writes the slots in first-appearance order to `s_slot`.
int order_by_first_row(pa_groupby* g, const uint32_t* c_first, const uint32_t* c_slot, uint32_t G, uint32_t* s_slot) {
  if (G == 0) return PA_OK;
  cudaStream_t st = g->stream;
  const uint64_t n_rows = static_cast<uint64_t>(std::max<int64_t>(g->n, 1));
  const uint64_t nblocks = (n_rows + 32ull * BM_BLOCK_WORDS - 1) / (32ull * BM_BLOCK_WORDS);
  const uint64_t nwords = nblocks * BM_BLOCK_WORDS;
  const uint32_t ntiles = static_cast<uint32_t>((nblocks + SC_TILE - 1) / SC_TILE);
  PA_TRY(g->scr.bitmap.alloc(nwords * 4, st));
  PA_TRY(g->scr.prefix8.alloc(nblocks * 4, st));
  PA_TRY(g->scr.tile_sums.alloc(static_cast<size_t>(ntiles) * 4, st));
  uint32_t* bitmap = g->scr.bitmap.as<uint32_t>();
  uint32_t* prefix8 = g->scr.prefix8.as<uint32_t>();
  uint32_t* tile_sums = g->scr.tile_sums.as<uint32_t>();
  CUDA_TRY(cudaMemsetAsync(bitmap, 0, nwords * 4, st));
  k_bm_set<<<(G + 255) / 256, 256, 0, st>>>(c_first, G, bitmap);
  CUDA_TRY(cudaGetLastError());
  const int cgrid = static_cast<int>(std::min<uint64_t>((nblocks + 255) / 256, static_cast<uint64_t>(g->num_sms) * 16));
  k_bm_count8<<<cgrid, 256, 0, st>>>(bitmap, nblocks, prefix8);
  CUDA_TRY(cudaGetLastError());
  k_scan_tiles<<<ntiles, 256, 0, st>>>(prefix8, nblocks, tile_sums);
  CUDA_TRY(cudaGetLastError());
  k_scan_sums<<<1, 256, 0, st>>>(tile_sums, ntiles);
  CUDA_TRY(cudaGetLastError());
  k_scan_apply<<<ntiles, 256, 0, st>>>(prefix8, nblocks, tile_sums);
  CUDA_TRY(cudaGetLastError());
  k_bm_rank<<<(G + 255) / 256, 256, 0, st>>>(c_first, c_slot, G, bitmap, prefix8, s_slot);
  CUDA_TRY(cudaGetLastError());
  g->last_launches += 6;
  return PA_OK;
}

// ------------------------------ global-table path ------------------------------

// device-wide exclusive scan of a uint32 array in place (order.cuh)
int scan_u32_on(pa_groupby* g, uint32_t* data, uint64_t n, DevBuf* tile_sums) {
  cudaStream_t st = g->stream;
  const uint32_t ntiles = static_cast<uint32_t>((n + SC_TILE - 1) / SC_TILE);
  PA_TRY(tile_sums->alloc(static_cast<size_t>(std::max<uint32_t>(ntiles, 1)) * 4, st));
  if (n == 0) return PA_OK;
  k_scan_tiles<<<ntiles, 256, 0, st>>>(data, n, tile_sums->as<uint32_t>());
  CUDA_TRY(cudaGetLastError());
  k_scan_sums<<<1, 256, 0, st>>>(tile_sums->as<uint32_t>(), ntiles);
  CUDA_TRY(cudaGetLastError());
  k_scan_apply<<<ntiles, 256, 0, st>>>(data, n, tile_sums->as<uint32_t>());
  CUDA_TRY(cudaGetLastError());
  return PA_OK;
}

// HyperLogLog estimate from the registers k_rp_hist1 filled (one key value in 2^HLL_SAMPLE_LOG2 feeds the sketch).
double hll_estimate(const uint32_t* reg) {
  const double m = HLL_M;
  double sum = 0;
  int zeros = 0;
  for (int i = 0; i < HLL_M; ++i) { sum += std::ldexp(1.0, -static_cast<int>(reg[i])); zeros += reg[i] == 0; }
  double e = (0.7213 / (1.0 + 1.079 / m)) * m * m / sum;
  if (e <= 2.5 * m && zeros > 0) e = m * std::log(m / zeros);      // small-range correction (linear counting)
  return e * static_cast<double>(1u << HLL_SAMPLE_LOG2);
}

// One partition level.  At 256 ways and more a 4096-row tile leaves runs of <= 16 rows (128-byte pieces of the key / value
// arrays, 64 of the row numbers): those take 8192-row tiles on one 1024-thread CTA per SM instead of two 512-thread CTAs
// with 4096-row tiles.  Measured per 1 B rows: 100 M groups (256 x 256) 45.0 -> 43.2 ms; at 128 ways the lost overlap
// between the two CTAs costs more than the longer runs give (16 M groups, 128 x 128: 32.0 -> 34.4 ms), so the threshold
// is 2^8.  PA_RP_BIG_TILE_LOG (environment, read once) moves it for A/B runs.
int launch_rp_scatter(pa_groupby* g, const RpArgs& a) {
  static const int big_from = [] { const char* e = std::getenv("PA_RP_BIG_TILE_LOG"); return e ? std::atoi(e) : 8; }();
  cudaStream_t st = g->stream;
  const bool nullable = !a.rows && a.vvalid;          // level 1 of a nullable value column: validity bit -> row-number word
  if (a.log_fan >= big_from) {
    auto kern = nullable ? k_rp_scatter_t<RP_THREADS_BIG, true> : k_rp_scatter_t<RP_THREADS_BIG, false>;
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(RpSmemBig::TOTAL)));
    kern<<<g->num_sms, RP_THREADS_BIG, RpSmemBig::TOTAL, st>>>(a);
  } else {
    auto kern = nullable ? k_rp_scatter_t<RP_THREADS, true> : k_rp_scatter_t<RP_THREADS, false>;
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(RpSmem::TOTAL)));
    kern<<<g->num_sms * 2, RP_THREADS, RpSmem::TOTAL, st>>>(a);
  }
  CUDA_TRY(cudaGetLastError());
  return PA_OK;
}

// The bucketed path (bucketed.cuh).  *declined = true: the estimate says a single shared-memory table holds the
// groups, or a bucket overflowed its table — the caller continues on the global-table path.
template <int VC, bool WIDE>
int run_bucketed_t(pa_groupby* g, const Column* val, uint32_t mask, uint64_t* cap_io, bool* declined, bool* table_filled) {
  using T = SmTab<VC, WIDE>;
  using SlotT = typename SlotOf<WIDE>::type;
  *table_filled = false;
  cudaStream_t st = g->stream;
  *declined = false;
  auto& sc = g->scr;
  const int64_t n = g->n;
  const uint64_t* keys = static_cast<const uint64_t*>(g->key_data);
  const uint64_t* vals = val ? static_cast<const uint64_t*>(val->data) : nullptr;
  CUDA_TRY(cudaEventRecord(g->ev[1], st));
  // ---- level 1 histogram (1024 fine buckets per chunk) + sketch ----
  // Everything up to the scatter depends on the KEYS only (the scatter keeps its cursors private), and a handle's keys
  // never change: histograms, offsets and bucket ends are computed by the first pass and reused by every later one.
  const uint32_t nchunks1 = static_cast<uint32_t>((n + RP_CHUNK_ROWS - 1) / RP_CHUNK_ROWS);
  CUDA_TRY(cudaMemsetAsync(g->status.p, 0, sizeof(uint32_t) * ST_WORDS, st));
  RpArgs a1{};
  a1.keys = keys; a1.vals = vals; a1.rows = nullptr; a1.n = n;
  a1.vvalid = val ? val->valid : nullptr; a1.voff = val ? val->bit_off : 0;
  a1.n_parents = 1; a1.n_chunks1 = nchunks1;
  if (!g->bk_have_hist) {
    PA_TRY(sc.rp_fine.alloc(sizeof(uint32_t) * RP_MAX_FAN * static_cast<size_t>(nchunks1), st));
    PA_TRY(sc.rp_hll.alloc(sizeof(uint32_t) * HLL_M, st));
    CUDA_TRY(cudaMemsetAsync(sc.rp_hll.p, 0, sizeof(uint32_t) * HLL_M, st));
    a1.counts = sc.rp_fine.as<unsigned int>(); a1.hll = sc.rp_hll.as<unsigned int>();
    k_rp_hist<true><<<g->num_sms * 2, RH_THREADS, 0, st>>>(a1);
    CUDA_TRY(cudaGetLastError());
    std::vector<uint32_t> reg(HLL_M);
    CUDA_TRY(cudaMemcpyAsync(reg.data(), sc.rp_hll.p, sizeof(uint32_t) * HLL_M, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    g->est_groups = hll_estimate(reg.data());
    g->bk_have_hist = true;
    g->bk_bits = g->bk_b1 = -1;
    g->last_launches += 1;
  }
  const double est = g->est_groups;
  const uint64_t hint = g->opt.expected_groups > 0 ? static_cast<uint64_t>(g->opt.expected_groups) : (g->have_groups ? g->G : 0);
  // plan for the larger of hint and estimate (the sketch is good to a few per cent; a wrong hint must not overflow the tables)
  const uint64_t plan = std::max<uint64_t>(hint, static_cast<uint64_t>(est * 1.05) + 64);
  if (!hint && plan <= static_cast<uint64_t>(T::CAP)) { *declined = true; return PA_OK; }   // the front table (gtable.cuh) holds them
  // Buckets of ~CAP/2 keys on average (the table admits 3/4 CAP; bucket sizes are Poisson around the mean).  Up to
  // 1024 buckets in one level; more = two levels with the bits split evenly (long runs in both scatters).
  const uint64_t per_bucket = T::CAP / 2;
  int bits = 1;
  while (bits < RP_MAX_BITS && (plan >> bits) > per_bucket) ++bits;
  int b1 = bits <= RP_SINGLE_MAX_LOG ? bits : (bits + 1) / 2;
  if (g->opt.bucket_bits > 0) {                         // tuning / test override: level-1 bits | level-2 bits << 8
    b1 = static_cast<int>(g->opt.bucket_bits & 0xFF);
    const int b2o = static_cast<int>((g->opt.bucket_bits >> 8) & 0xFF);
    if (b1 < 1 || b1 > RP_L1_LOG || b2o > RP_L1_LOG) return set_err(PA_ERR_INVALID, "bucket bits override out of range");
    bits = b1 + b2o;
  }
  const int b2 = bits - b1;
  const uint32_t nb = 1u << bits;
  const size_t pad = 4;
  const bool replan = g->bk_bits != bits || g->bk_b1 != b1;    // (first pass, or the group-count hint moved the plan)
  // ---- level 1: fold the fine counts to 2^b1 buckets, scan, bucket ends, scatter ----
  const size_t flat1 = (static_cast<size_t>(nchunks1) << b1) + 1;
  if (replan) {
    PA_TRY(sc.rp_counts1.alloc(sizeof(uint32_t) * flat1, st));
    PA_TRY(sc.rp_ends1.alloc(sizeof(uint32_t) * (1u << b1), st));
    CUDA_TRY(cudaMemsetAsync(sc.rp_counts1.as<uint32_t>() + (flat1 - 1), 0, sizeof(uint32_t), st));
    k_rp_fold<<<static_cast<unsigned>((flat1 - 1 + 255) / 256), 256, 0, st>>>(sc.rp_fine.as<unsigned int>(), nchunks1, b1, sc.rp_counts1.as<unsigned int>());
    CUDA_TRY(cudaGetLastError());
    PA_TRY(scan_u32_on(g, sc.rp_counts1.as<uint32_t>(), flat1, &sc.tile_sums));
    g->last_launches += 4;
  }
  PA_TRY(sc.p_keys.alloc((static_cast<size_t>(n) + pad) * 8, st));
  if (vals) PA_TRY(sc.p_vals.alloc((static_cast<size_t>(n) + pad) * 8, st));
  PA_TRY(sc.p_rows.alloc((static_cast<size_t>(n) + pad) * 4, st));
  a1.shift = 64 - b1; a1.log_fan = b1;
  a1.offsets = sc.rp_counts1.as<unsigned int>();
  a1.out_keys = sc.p_keys.as<uint64_t>(); a1.out_vals = vals ? sc.p_vals.as<uint64_t>() : nullptr; a1.out_rows = sc.p_rows.as<uint32_t>();
  if (replan) {
    k_rp_ends<<<((1u << b1) + 255) / 256, 256, 0, st>>>(a1, sc.rp_ends1.as<unsigned int>());
    CUDA_TRY(cudaGetLastError());
    g->last_launches += 1;
  }
  PA_TRY(launch_rp_scatter(g, a1));
  g->last_launches += 1;
  BkArgs b{};
  b.keys = sc.p_keys.as<uint64_t>(); b.vals = vals ? sc.p_vals.as<uint64_t>() : nullptr; b.rows = sc.p_rows.as<uint32_t>();
  b.bucket_end = sc.rp_ends1.as<unsigned int>();
  b.nullable = (val && val->valid) ? 1 : 0;
  if (b2 > 0) {
    // ---- level 2 inside every level-1 bucket ----
    const int np = 1 << b1;
    const size_t chunks2_max = static_cast<size_t>(n) / RP_CHUNK_ROWS + np + 1;
    const size_t flat2 = (chunks2_max << b2) + 1;
    // (Only level 1 is cached: inside a tile's run the level-1 scatter orders rows by atomic arrival, so the rows on
    // either side of a level-2 chunk boundary differ from pass to pass and the level-2 counts have to be retaken.)
    PA_TRY(sc.rp_tiles.alloc(sizeof(uint32_t) * (np + 1), st));
    PA_TRY(sc.rp_counts2.alloc(sizeof(uint32_t) * flat2, st));
    PA_TRY(sc.rp_ends2.alloc(sizeof(uint32_t) * nb, st));
    CUDA_TRY(cudaMemsetAsync(sc.rp_counts2.p, 0, sizeof(uint32_t) * flat2, st));
    if (replan) {
      k_rp_cprefix<<<1, 1024, 0, st>>>(sc.rp_ends1.as<unsigned int>(), np, sc.rp_tiles.as<unsigned int>());
      CUDA_TRY(cudaGetLastError());
    }
    RpArgs a2{};
    a2.keys = sc.p_keys.as<uint64_t>(); a2.vals = b.vals; a2.rows = sc.p_rows.as<uint32_t>(); a2.n = n;
    a2.shift = 64 - bits; a2.log_fan = b2; a2.n_parents = np;
    a2.parent_end = sc.rp_ends1.as<unsigned int>(); a2.cprefix = sc.rp_tiles.as<unsigned int>();
    a2.counts = sc.rp_counts2.as<unsigned int>();
    k_rp_hist<false><<<g->num_sms * 2, RH_THREADS, 0, st>>>(a2);
    CUDA_TRY(cudaGetLastError());
    PA_TRY(scan_u32_on(g, sc.rp_counts2.as<uint32_t>(), flat2, &sc.tile_sums));
    g->last_launches += 5;
    PA_TRY(sc.q_keys.alloc((static_cast<size_t>(n) + pad) * 8, st));
    if (vals) PA_TRY(sc.q_vals.alloc((static_cast<size_t>(n) + pad) * 8, st));
    PA_TRY(sc.q_rows.alloc((static_cast<size_t>(n) + pad) * 4, st));
    a2.offsets = sc.rp_counts2.as<unsigned int>();
    a2.out_keys = sc.q_keys.as<uint64_t>(); a2.out_vals = vals ? sc.q_vals.as<uint64_t>() : nullptr; a2.out_rows = sc.q_rows.as<uint32_t>();
    k_rp_ends<<<(nb + 255) / 256, 256, 0, st>>>(a2, sc.rp_ends2.as<unsigned int>());
    CUDA_TRY(cudaGetLastError());
    g->last_launches += 1;
    PA_TRY(launch_rp_scatter(g, a2));
    g->last_launches += 1;
    b.keys = sc.q_keys.as<uint64_t>(); b.vals = vals ? sc.q_vals.as<uint64_t>() : nullptr; b.rows = sc.q_rows.as<uint32_t>();
    b.bucket_end = sc.rp_ends2.as<unsigned int>();
  }
  g->bk_bits = bits; g->bk_b1 = b1;
  // ---- bucket aggregation ----
  // Few buckets (they would leave SMs idle, and a bucket is as long as its keys are frequent): ranged mode — equal
  // row shares per CTA, tables flushed into the global table, which the caller then compacts and orders as usual.
  const bool ranged = nb < static_cast<uint32_t>(4 * g->num_sms);
  BkArgs& bref = b;
  bref.ranged = ranged ? 1 : 0;
  bref.n = n;
  if (ranged) {
    uint64_t cap = *cap_io;
    while (cap < plan * 2) cap <<= 1;
    *cap_io = cap;
    const uint64_t nslots = cap + 2;
    PA_TRY(sc.table.alloc(nslots * sizeof(SlotT), st));
    const int init_grid = static_cast<int>(std::min<uint64_t>((nslots + 255) / 256, static_cast<uint64_t>(g->num_sms) * 16));
    k_gtable_init<WIDE><<<init_grid, 256, 0, st>>>(sc.table.as<SlotT>(), nslots);
    CUDA_TRY(cudaGetLastError());
    bref.table = sc.table.p; bref.cap_mask = cap - 1; bref.shift = 64 - __builtin_ctzll(cap);
    bref.n_buckets = nb; bref.part_bits = bits; bref.agg_mask = mask; bref.max_keys = T::MAX_KEYS;
    bref.status = g->status.as<uint32_t>();
    auto kern = bref.nullable ? k_bucket_agg<VC, WIDE, true> : k_bucket_agg<VC, WIDE, false>;
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(T::TOTAL)));
    kern<<<g->num_sms, BK_THREADS, T::TOTAL, st>>>(bref);
    CUDA_TRY(cudaGetLastError());
    g->last_launches += 2;
    uint32_t h_status[ST_WORDS];
    CUDA_TRY(cudaMemcpyAsync(h_status, g->status.p, sizeof h_status, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (h_status[ST_OVERFLOW]) { *declined = true; return PA_OK; }
    g->last_mode = 5;
    g->last_rlog = bits;
    *table_filled = true;
    return PA_OK;
  }
  uint64_t u_cap64 = std::min<uint64_t>(static_cast<uint64_t>(n) + 1, plan + plan / 4 + 65536);
  u_cap64 = std::min<uint64_t>(u_cap64, static_cast<uint64_t>(nb) * (T::MAX_KEYS + 1));
  const uint32_t u_cap = static_cast<uint32_t>(std::min<uint64_t>(u_cap64, 0xFFFFFFF0ull));
  using Rec = typename BkRecOf<WIDE>::type;
  PA_TRY(sc.u_rec.alloc(static_cast<size_t>(u_cap) * sizeof(Rec), st));
  PA_TRY(sc.u_first.alloc(static_cast<size_t>(u_cap) * 4, st));
  PA_TRY(sc.rp_next.alloc(4, st));
  CUDA_TRY(cudaMemsetAsync(sc.rp_next.p, 0, 4, st));
  b.n_buckets = nb; b.part_bits = bits; b.next_bucket = sc.rp_next.as<unsigned int>();
  b.agg_mask = mask; b.max_keys = T::MAX_KEYS;
  b.u_rec = sc.u_rec.p; b.u_first = sc.u_first.as<uint32_t>();
  b.u_cap = u_cap; b.status = g->status.as<uint32_t>();
  {
    auto kern = b.nullable ? k_bucket_agg<VC, WIDE, true> : k_bucket_agg<VC, WIDE, false>;
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(T::TOTAL)));
    kern<<<g->num_sms, BK_THREADS, T::TOTAL, st>>>(b);
    CUDA_TRY(cudaGetLastError());
  }
  g->last_launches += 1;
  CUDA_TRY(cudaEventRecord(g->ev[2], st));
  uint32_t h_status[ST_WORDS];
  CUDA_TRY(cudaMemcpyAsync(h_status, g->status.p, sizeof h_status, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  if (h_status[ST_OVERFLOW]) { *declined = true; return PA_OK; }
  const uint32_t G = h_status[ST_COUNTER];
  if (!WIDE && g->want_unordered) {   // the sharded step exports the records as they are (see pa_groupby::want_unordered)
    g->unordered = true;
    g->unordered_recs = sc.u_rec.p;
    g->unordered_G = G;
    g->last_mode = 5;
    g->last_rlog = bits;
    CUDA_TRY(cudaEventRecord(g->ev[3], st));
    return PA_OK;
  }
  g->G = G;
  PA_TRY(alloc_result(g, G, WIDE, VC != VC_F));
  if (G > 0) {
    // ---- first-appearance order by bitmap rank, written straight into the GroupResult ----
    const uint64_t n_rows = static_cast<uint64_t>(std::max<int64_t>(n, 1));
    const uint64_t nblocks = (n_rows + 32ull * BM_BLOCK_WORDS - 1) / (32ull * BM_BLOCK_WORDS);
    const uint64_t nwords = nblocks * BM_BLOCK_WORDS;
    const uint32_t ntiles = static_cast<uint32_t>((nblocks + SC_TILE - 1) / SC_TILE);
    PA_TRY(sc.bitmap.alloc(nwords * 4, st));
    PA_TRY(sc.prefix8.alloc(nblocks * 4, st));
    PA_TRY(sc.tile_sums.alloc(static_cast<size_t>(std::max<uint32_t>(ntiles, 1)) * 4, st));
    CUDA_TRY(cudaMemsetAsync(sc.bitmap.p, 0, nwords * 4, st));
    k_bm_set<<<(G + 255) / 256, 256, 0, st>>>(b.u_first, G, sc.bitmap.as<uint32_t>());
    CUDA_TRY(cudaGetLastError());
    const int cgrid = static_cast<int>(std::min<uint64_t>((nblocks + 255) / 256, static_cast<uint64_t>(g->num_sms) * 16));
    k_bm_count8<<<cgrid, 256, 0, st>>>(sc.bitmap.as<uint32_t>(), nblocks, sc.prefix8.as<uint32_t>());
    CUDA_TRY(cudaGetLastError());
    k_scan_tiles<<<ntiles, 256, 0, st>>>(sc.prefix8.as<uint32_t>(), nblocks, sc.tile_sums.as<uint32_t>());
    CUDA_TRY(cudaGetLastError());
    k_scan_sums<<<1, 256, 0, st>>>(sc.tile_sums.as<uint32_t>(), ntiles);
    CUDA_TRY(cudaGetLastError());
    k_scan_apply<<<ntiles, 256, 0, st>>>(sc.prefix8.as<uint32_t>(), nblocks, sc.tile_sums.as<uint32_t>());
    CUDA_TRY(cudaGetLastError());
    PA_TRY(sc.s_slot.alloc(static_cast<size_t>(G) * 4, st));
    k_bm_rank<<<(G + 255) / 256, 256, 0, st>>>(b.u_first, nullptr, G, sc.bitmap.as<uint32_t>(), sc.prefix8.as<uint32_t>(), sc.s_slot.as<uint32_t>());
    CUDA_TRY(cudaGetLastError());
    k_bk_gather<WIDE><<<(G + 255) / 256, 256, 0, st>>>(sc.u_rec.p, sc.s_slot.as<uint32_t>(), G, g->res);
    CUDA_TRY(cudaGetLastError());
    g->last_launches += 1;
    g->last_launches += 6;
  }
  g->last_mode = 5;
  g->last_rlog = bits;
  CUDA_TRY(cudaEventRecord(g->ev[3], st));
  return PA_OK;
}

template <int VC, bool WIDE>
int run_global_t(pa_groupby* g, const Column* val, uint32_t mask) {
  using SlotT = typename SlotOf<WIDE>::type;
  cudaStream_t st = g->stream;
  // (an earlier pass on this handle knows the group count exactly: size for it instead of regrowing every call)
  uint64_t want = g->opt.expected_groups > 0 ? static_cast<uint64_t>(g->opt.expected_groups)
                  : (g->have_groups ? std::max<uint64_t>(g->G, 1) : std::min<uint64_t>(static_cast<uint64_t>(g->n), 1ull << 20));
  // Load factor <= 1/2, and never fewer than n / 64 slots (at most 2 M): a small group count
  // hint must not buy a small, crowded table (scattered keys: 30 000 groups in 65 536 slots measured 27 ms
  // per 1 B rows against 21.6 ms in 2 M slots — longer probe sequences, more contended sectors).
  uint64_t cap = 1024;
  const uint64_t cap_floor = std::min<uint64_t>(2ull << 20, static_cast<uint64_t>(g->n) / 64);
  while (cap < want * 2 || cap < cap_floor) cap <<= 1;
  const uint64_t cap_limit = [&] { uint64_t c = 1024; while (c < static_cast<uint64_t>(g->n) * 2) c <<= 1; return c; }();
  if (cap > cap_limit) cap = cap_limit;
  DevBuf& table = g->scr.table;
  const int grid_full = g->num_sms * 6;   // two waves of the 3 resident CTAs per SM
  bool table_filled = false;              // the bucketed path (ranged mode) already left the groups in `table`
  {
    // More groups than one shared-memory table holds (or nobody knows how many): partition into buckets and
    // aggregate those in shared memory (bucketed.cuh); it declines when its own estimate says the front table is enough
    const uint64_t known0 = g->opt.expected_groups > 0 ? static_cast<uint64_t>(g->opt.expected_groups) : (g->have_groups ? g->G : 0);
    // (a nullable VALUE column is fine below 2^31 rows: the validity bit rides in the row-number word of the partition)
    const bool plain = g->key_width == 8 && (!val || val->width == 8) && !g->key_valid && (!val || !val->valid || g->n < (1ll << 31)) &&
                       reinterpret_cast<uintptr_t>(g->key_data) % 32 == 0 && (!val || reinterpret_cast<uintptr_t>(val->data) % 32 == 0);
    if (plain && !g->opt.no_partition && g->n >= (1ll << 22) && (known0 == 0 || known0 > static_cast<uint64_t>(SmTab<VC, WIDE>::CAP))) {
      bool declined = false;
      PA_TRY((run_bucketed_t<VC, WIDE>(g, val, mask, &cap, &declined, &table_filled)));
      if (!declined && !table_filled) return PA_OK;
      if (declined) { g->last_mode = 0; g->last_rlog = 0; }
    }
  }
  if (!table_filled) CUDA_TRY(cudaEventRecord(g->ev[1], st));
  while (!table_filled) {
    const uint64_t nslots = cap + 2;
    PA_TRY(table.alloc(nslots * sizeof(SlotT), st));
    CUDA_TRY(cudaMemsetAsync(g->status.p, 0, sizeof(uint32_t) * ST_WORDS, st));
    const int init_grid = static_cast<int>(std::min<uint64_t>((nslots + 255) / 256, static_cast<uint64_t>(g->num_sms) * 16));
    k_gtable_init<WIDE><<<init_grid, 256, 0, st>>>(table.as<SlotT>(), nslots);
    CUDA_TRY(cudaGetLastError());
    GScanArgs a{};
    a.keys = g->key_data;
    a.kvalid = g->key_valid;
    a.koff = g->key_bit_off;
    a.kw = g->key_width;
    a.vals = val ? val->data : nullptr;
    a.vvalid = val ? val->valid : nullptr;
    a.voff = val ? val->bit_off : 0;
    a.vw = val ? val->width : 8;
    a.n = g->n;
    a.table = table.p;
    a.cap_mask = cap - 1;
    a.shift = 64 - __builtin_ctzll(cap);
    a.status = g->status.as<uint32_t>();
    a.agg_mask = mask;
    const int64_t ntiles = (g->n + 1023) / 1024;
    const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(ntiles, grid_full)));
    const bool fast = a.kw == 8 && (!a.vals || a.vw == 8) && !a.kvalid &&
                      reinterpret_cast<uintptr_t>(a.keys) % 32 == 0 && reinterpret_cast<uintptr_t>(a.vals) % 32 == 0;
    // Very many groups (table far larger than L2): reorder the rows by table region first (partition.cuh).
    DevBuf &p_keys = g->scr.p_keys, &p_vals = g->scr.p_vals, &p_rows = g->scr.p_rows, &p_counts = g->scr.p_counts;
    const uint64_t known_g = g->opt.expected_groups > 0 ? static_cast<uint64_t>(g->opt.expected_groups) : (g->have_groups ? g->G : 0);
    if (fast && a.vals && !a.vvalid && known_g >= (2ull << 20) && g->n >= (1ll << 22) && !g->opt.no_partition) {
      const uint64_t table_bytes = nslots * sizeof(SlotT);
      int log_parts = 6;
      while (log_parts < 10 && (table_bytes >> log_parts) > (16ull << 20)) ++log_parts;
      const int parts = 1 << log_parts;
      PA_TRY(p_keys.alloc(static_cast<size_t>(g->n) * 8, st));
      PA_TRY(p_vals.alloc(static_cast<size_t>(g->n) * 8, st));
      PA_TRY(p_rows.alloc(static_cast<size_t>(g->n) * 4, st));
      PA_TRY(p_counts.alloc(sizeof(unsigned long long) * parts, st));
      CUDA_TRY(cudaMemsetAsync(p_counts.p, 0, sizeof(unsigned long long) * parts, st));
      PartArgs pa_{};
      pa_.keys = static_cast<const uint64_t*>(a.keys);
      pa_.vals = static_cast<const uint64_t*>(a.vals);
      pa_.n = g->n;
      pa_.log_parts = log_parts;
      pa_.counts = p_counts.as<unsigned long long>();
      pa_.out_keys = p_keys.as<uint64_t>();
      pa_.out_vals = p_vals.as<uint64_t>();
      pa_.out_rows = p_rows.as<uint32_t>();
      k_part_hist<<<g->num_sms * 2, PH_THREADS, 0, st>>>(pa_);
      CUDA_TRY(cudaGetLastError());
      k_part_offsets<<<1, PT_MAX_PARTS, 0, st>>>(pa_.counts, parts);
      CUDA_TRY(cudaGetLastError());
      CUDA_TRY(cudaFuncSetAttribute(k_part_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(PtSmem::TOTAL)));
      k_part_scatter<<<g->num_sms * 2, PT_THREADS, PtSmem::TOTAL, st>>>(pa_);
      CUDA_TRY(cudaGetLastError());
      g->last_launches += 3;
      a.keys = p_keys.p;
      a.vals = p_vals.p;
      a.rowids = p_rows.as<uint32_t>();
      g->last_rlog = log_parts;   // reported through pa_groupby_last_detail[1] on this path
    }
    // Shared-memory front table unless the caller (or an earlier pass on this handle) says there are
    // far more groups than it holds; it spills to the global table, so it is correct for any input.
    const uint64_t known = g->opt.expected_groups > 0 ? static_cast<uint64_t>(g->opt.expected_groups) : (g->have_groups ? g->G : 0);
    const bool front = known <= static_cast<uint64_t>(SmTab<VC, WIDE>::CAP);   // (dense keys fill every slot; hashed keys 3/4)
    a.sm_max_keys = static_cast<uint32_t>(SmTab<VC, WIDE>::MAX_KEYS);
    DevBuf& krange = g->scr.krange;
    if (front) {
      PA_TRY(krange.alloc(sizeof(KeyRange), st));
      CUDA_TRY(cudaMemsetAsync(krange.p, 0, sizeof(KeyRange), st));
      a.krange = krange.as<KeyRange>();
      k_key_range<<<SM_SAMPLE_GRID, 256, 0, st>>>(a);
      CUDA_TRY(cudaGetLastError());
      g->last_launches += 1;
      auto kern = fast ? k_smemtab_scan<VC, WIDE, true> : k_smemtab_scan<VC, WIDE, false>;
      const size_t smem = SmTab<VC, WIDE>::TOTAL;
      CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
      kern<<<g->num_sms, SM_THREADS, smem, st>>>(a);
    } else if (fast) {
      k_gtable_scan<VC, WIDE, true><<<grid, 256, 0, st>>>(a);
    } else {
      k_gtable_scan<VC, WIDE, false><<<grid, 256, 0, st>>>(a);
    }
    g->last_mode = front ? 3 : (a.rowids ? 4 : 0);
    CUDA_TRY(cudaGetLastError());
    g->last_launches += 2;
    uint32_t h_status[ST_WORDS];
    CUDA_TRY(cudaMemcpyAsync(h_status, g->status.p, sizeof h_status, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (!h_status[ST_OVERFLOW]) break;
    if (cap >= cap_limit) return set_err(PA_ERR_CUDA, "global group table overflowed at capacity %llu", (unsigned long long)cap);
    cap = std::min(cap * 8, cap_limit);
  }
  CUDA_TRY(cudaEventRecord(g->ev[2], st));
  // compact occupied slots, order them by first row, gather
  const uint64_t nslots = cap + 2;
  const uint64_t max_groups = std::min<uint64_t>(nslots, static_cast<uint64_t>(g->n) + 2);
  DevBuf &c_first = g->scr.c_first, &c_slot = g->scr.c_slot, &s_slot = g->scr.s_slot;
  PA_TRY(c_first.alloc(max_groups * 4, st));
  PA_TRY(c_slot.alloc(max_groups * 4, st));
  const int cgrid = static_cast<int>(std::min<uint64_t>((nslots + 255) / 256, static_cast<uint64_t>(g->num_sms) * 16));
  k_gtable_compact<WIDE><<<cgrid, 256, 0, st>>>(table.as<SlotT>(), nslots, c_first.as<uint32_t>(), c_slot.as<uint32_t>(), g->status.as<uint32_t>());
  CUDA_TRY(cudaGetLastError());
  g->last_launches += 1;
  uint32_t G = 0;
  CUDA_TRY(cudaMemcpyAsync(&G, g->status.as<uint32_t>() + ST_COUNTER, 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  g->G = G;
  PA_TRY(alloc_result(g, G, WIDE, VC != VC_F));
  if (G > 0) {
    PA_TRY(s_slot.alloc(static_cast<size_t>(G) * 4, st));
    PA_TRY(order_by_first_row(g, c_first.as<uint32_t>(), c_slot.as<uint32_t>(), G, s_slot.as<uint32_t>()));
    k_gtable_gather<WIDE><<<(G + 255) / 256, 256, 0, st>>>(table.as<SlotT>(), cap, s_slot.as<uint32_t>(), G, g->res);
    CUDA_TRY(cudaGetLastError());
    g->last_launches += 1;
  }
  CUDA_TRY(cudaEventRecord(g->ev[3], st));
  return PA_OK;
}

int run_global(pa_groupby* g, const Column* val, uint32_t mask, bool wide) {
  const int vc = val ? val->vc : VC_I;
  if (wide) {
    if (vc == VC_F) return run_global_t<VC_F, true>(g, val, mask);
    if (vc == VC_I) return run_global_t<VC_I, true>(g, val, mask);
    return run_global_t<VC_U, true>(g, val, mask);
  }
  if (vc == VC_F) return run_global_t<VC_F, false>(g, val, mask);
  if (vc == VC_I) return run_global_t<VC_I, false>(g, val, mask);
  return run_global_t<VC_U, false>(g, val, mask);
}

// ------------------------------ emit ------------------------------
const char* sum_format(int vc) { return vc == VC_F ? "g" : (vc == VC_I ? "l" : "L"); }

int run_emit(pa_groupby* g, const Column* val, uint32_t mask) {
  cudaStream_t st = g->stream;
  g->outs.clear();
  const uint32_t G = g->G;
  const size_t words = (static_cast<size_t>(G) + 31) / 32 + 1;
  EmitArgs e{};
  e.r = g->res;
  e.G = G;
  e.G_dev = g->emit_G_dev;
  e.vc = val ? val->vc : VC_I;
  e.vw = val ? val->width : 8;
  e.vals = val ? val->data : nullptr;
  e.vvalid = val ? val->valid : nullptr;
  e.voff = val ? val->bit_off : 0;
  if (g->merged) {
    e.vc = g->last_vc; e.vw = g->last_vw;
    e.m_first_val = g->m_first_val.as<uint64_t>(); e.m_last_val = g->m_last_val.as<uint64_t>();
    e.m_first_valid = g->m_first_valid.as<uint8_t>(); e.m_last_valid = g->m_last_valid.as<uint8_t>();
  }
  auto add = [&](uint32_t bit, const std::string& fmt, int width, bool nullable, void** vptr, uint32_t** bptr) -> int {
    g->outs.emplace_back();
    AggOut& o = g->outs.back();
    o.bit = bit;
    o.format = fmt;
    o.width = width;
    o.nullable = nullable;
    PA_TRY(o.values.alloc(static_cast<size_t>(std::max<uint32_t>(G, 1)) * width, st));
    *vptr = o.values.p;
    if (nullable) {
      PA_TRY(o.valid.alloc(words * 4, st));
      *bptr = o.valid.as<uint32_t>();
    }
    return PA_OK;
  };
  g->outs.reserve(8);
  void* v;
  uint32_t* b;
  const std::string vfmt = g->merged ? g->last_vfmt : (val ? val->format : "l");
  if (mask & AGG_SUM) { PA_TRY(add(AGG_SUM, sum_format(e.vc), 8, true, &v, &b)); e.o_sum = v; e.o_sum_valid = b; }
  if (mask & AGG_MEAN) { PA_TRY(add(AGG_MEAN, "g", 8, true, &v, &b)); e.o_mean = static_cast<double*>(v); e.o_mean_valid = b; }
  if (mask & AGG_COUNT) { PA_TRY(add(AGG_COUNT, "l", 8, false, &v, &b)); e.o_count = static_cast<int64_t*>(v); }
  if (mask & AGG_MIN) { PA_TRY(add(AGG_MIN, vfmt, e.vw, true, &v, &b)); e.o_min = v; e.o_min_valid = b; }
  if (mask & AGG_MAX) { PA_TRY(add(AGG_MAX, vfmt, e.vw, true, &v, &b)); e.o_max = v; e.o_max_valid = b; }
  if (mask & AGG_FIRST) { PA_TRY(add(AGG_FIRST, vfmt, e.vw, true, &v, &b)); e.o_first = v; e.o_first_valid = b; }
  if (mask & AGG_LAST) { PA_TRY(add(AGG_LAST, vfmt, e.vw, true, &v, &b)); e.o_last = v; e.o_last_valid = b; }
  if (G > 0 && mask) {
    k_emit<<<(G + 255) / 256, 256, 0, st>>>(e);
    CUDA_TRY(cudaGetLastError());
    g->last_launches += 1;
  }
  return PA_OK;
}

// ------------------------------ key -> group id lookup, second-stage aggregates ------------------------------
// Read-only open-addressing table key -> rank (first-appearance order) built from the finished GroupResult.
struct RowLookup {
  DevBuf tkeys, tranks, special;
  RowIdArgs a{};
};

int build_row_lookup(pa_groupby* g, RowLookup* lk) {
  cudaStream_t st = g->stream;
  const uint32_t G = g->G;
  uint64_t cap = 1024;
  while (cap < static_cast<uint64_t>(G) * 2) cap <<= 1;
  PA_TRY(lk->tkeys.alloc(cap * 8, st));
  PA_TRY(lk->tranks.alloc(cap * 4, st));
  PA_TRY(lk->special.alloc(8, st));
  const int fgrid = static_cast<int>(std::min<uint64_t>((cap + 255) / 256, static_cast<uint64_t>(g->num_sms) * 16));
  k_fill_u64<<<fgrid, 256, 0, st>>>(lk->tkeys.as<unsigned long long>(), cap, kEmptyKey);
  CUDA_TRY(cudaMemsetAsync(lk->special.p, 0xFF, 8, st));
  RowIdArgs& a = lk->a;
  a.tkeys = lk->tkeys.as<unsigned long long>();
  a.tranks = lk->tranks.as<uint32_t>();
  a.cap_mask = cap - 1;
  a.shift = 64 - __builtin_ctzll(cap);
  a.special = lk->special.as<uint32_t>();
  a.gkey = g->res.key;
  a.gkind = g->res.key_kind;
  a.G = G;
  a.keys = g->key_data;
  a.kvalid = g->key_valid;
  a.koff = g->key_bit_off;
  a.kw = g->key_width;
  a.n = g->n;
  a.resample = g->resample ? 1 : 0;
  a.rs = g->rs;
  a.out = nullptr;
  if (G) {
    k_rowid_build<<<(G + 255) / 256, 256, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
  }
  return PA_OK;
}

// The key columns of a hashed key, as k_row_hash / k_row_verify read them
RowKeys row_keys(const pa_groupby* g) {
  RowKeys k{};
  k.n_cols = static_cast<int>(g->keys.size());
  k.n = g->n;
  for (int j = 0; j < k.n_cols; ++j) {
    const Column& c = g->keys[j];
    k.valid[j] = c.valid;
    k.off[j] = c.bit_off;
    if (c.is_str) k.str[j] = c.str;
    else { k.col[j] = c.data; k.width[j] = c.width; }
  }
  return k;
}

// Every row of a hashed key against its group's first row (k_row_verify); *collided: two different keys share a hash
int verify_hashed_keys(pa_groupby* g, bool* collided) {
  cudaStream_t st = g->stream;
  *collided = false;
  if (g->n == 0 || g->G == 0) return PA_OK;
  RowLookup lk;
  PA_TRY(build_row_lookup(g, &lk));
  DevBuf flag;
  PA_TRY(flag.alloc(4, st));
  CUDA_TRY(cudaMemsetAsync(flag.p, 0, 4, st));
  const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((g->n + 255) / 256, static_cast<int64_t>(g->num_sms) * 16)));
  k_row_verify<<<grid, 256, 0, st>>>(row_keys(g), lk.a, g->res.first_row, flag.as<uint32_t>());
  CUDA_TRY(cudaGetLastError());
  uint32_t h = 0;
  CUDA_TRY(cudaMemcpyAsync(&h, flag.p, 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  if (h == 2u) return set_err(PA_ERR_STATE, "%s: a row's hash is missing from the group table", g->keys.size() == 1 ? "utf8 keys" : "hashed composite key");
  *collided = h != 0;
  return PA_OK;
}

// Outputs of product / variance / stddev (k_stage2_emit) from the per-group terms on the handle (g->s2_m2 / s2_prod):
// after the second pass on a rank's rows, or after the merge of stage-2 records.  Appends them to g->outs.
int emit_stage2(pa_groupby* g, int vc, uint32_t ext) {
  cudaStream_t st = g->stream;
  const uint32_t G = g->G;
  const size_t words = (static_cast<size_t>(G) + 31) / 32 + 1;
  const size_t gbytes = static_cast<size_t>(std::max<uint32_t>(G, 1)) * 8;
  Stage2Emit e{};
  e.r = g->res;
  e.G = G;
  e.vc = vc;
  e.m2 = (ext & (AGG_VARIANCE | AGG_STDDEV)) ? g->s2_m2.as<double>() : nullptr;
  e.prod = (ext & AGG_PRODUCT) ? g->s2_prod.as<unsigned long long>() : nullptr;
  auto add = [&](uint32_t bit, const std::string& fmt, void** vptr, uint32_t** bptr) -> int {
    g->outs.emplace_back();
    AggOut& o = g->outs.back();
    o.bit = bit;
    o.format = fmt;
    o.width = 8;
    o.nullable = true;
    PA_TRY(o.values.alloc(gbytes, st));
    PA_TRY(o.valid.alloc(words * 4, st));
    *vptr = o.values.p;
    *bptr = o.valid.as<uint32_t>();
    return PA_OK;
  };
  void* v;
  uint32_t* b;
  if (ext & AGG_PRODUCT) { PA_TRY(add(AGG_PRODUCT, sum_format(vc), &v, &b)); e.o_prod = static_cast<unsigned long long*>(v); e.o_prod_valid = b; }
  if (ext & AGG_VARIANCE) { PA_TRY(add(AGG_VARIANCE, "g", &v, &b)); e.o_var = static_cast<double*>(v); e.o_var_valid = b; }
  if (ext & AGG_STDDEV) { PA_TRY(add(AGG_STDDEV, "g", &v, &b)); e.o_std = static_cast<double*>(v); e.o_std_valid = b; }
  if (G == 0) return PA_OK;
  k_stage2_emit<<<(G + 255) / 256, 256, 0, st>>>(e);
  CUDA_TRY(cudaGetLastError());
  return PA_OK;
}

// product / variance / stddev (stage2.cuh): the second pass over keys + values, after the ordinary pass has
// produced sum (or the double sum) and count per group.  Appends its outputs to g->outs; the per-group M2 / product stay
// on the handle (g->s2_m2 / s2_prod) until the next aggregate.
int run_stage2(pa_groupby* g, const Column* val, uint32_t ext) {
  cudaStream_t st = g->stream;
  const uint32_t G = g->G;
  const int vc = val->vc;
  const bool want_m2 = (ext & (AGG_VARIANCE | AGG_STDDEV)) != 0, want_prod = (ext & AGG_PRODUCT) != 0;
  DevBuf mean;
  const size_t gbytes = static_cast<size_t>(std::max<uint32_t>(G, 1)) * 8;
  PA_TRY(mean.alloc(gbytes, st));
  if (want_m2) PA_TRY(g->s2_m2.alloc(gbytes, st)); else g->s2_m2.reset();
  if (want_prod) PA_TRY(g->s2_prod.alloc(gbytes, st)); else g->s2_prod.reset();
  double* m2 = want_m2 ? g->s2_m2.as<double>() : nullptr;
  unsigned long long* prod = want_prod ? g->s2_prod.as<unsigned long long>() : nullptr;
  g->s2_ext = ext;
  if (G == 0) return emit_stage2(g, vc, ext);
  RowLookup lk;
  PA_TRY(build_row_lookup(g, &lk));
  k_stage2_init<<<(G + 255) / 256, 256, 0, st>>>(g->res, G, vc, mean.as<double>(), m2, prod);
  CUDA_TRY(cudaGetLastError());
  Stage2Args a{};
  a.ids = lk.a;
  a.vals = val->data;
  a.vvalid = val->valid;
  a.voff = val->bit_off;
  a.vw = val->width;
  a.mean = mean.as<double>();
  a.m2 = m2;
  a.prod = prod;
  a.use_smem = G <= S2_SMEM_SLOTS ? 1u : 0u;
  a.rlog = 0;
  // (replicas only while they stay small: the key -> id lookups want the L1 that shared memory takes away —
  //  1000 groups measured 5.7 ms per 1 B rows unreplicated against 7.3 ms with 4 replicas)
  while (a.use_smem && a.rlog < 5 && (static_cast<uint64_t>(G) << (a.rlog + 1)) <= S2_REPL_SLOTS) ++a.rlog;
  if (g->n > 0) {
    const size_t smem = a.use_smem ? (static_cast<size_t>(G) << a.rlog) * 16 : 0;
    auto kern = vc == VC_F ? k_stage2<VC_F> : (vc == VC_I ? k_stage2<VC_I> : k_stage2<VC_U>);
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(S2_SMEM_SLOTS * 16)));
    int per_sm = 1;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, S2_THREADS, smem));
    const int64_t want = (g->n + S2_THREADS - 1) / S2_THREADS;
    const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(want, static_cast<int64_t>(g->num_sms) * std::max(per_sm, 1))));
    kern<<<grid, S2_THREADS, smem, st>>>(a);
    CUDA_TRY(cudaGetLastError());
  }
  PA_TRY(emit_stage2(g, vc, ext));
  g->last_launches += 5;
  CUDA_TRY(cudaEventRecord(g->ev[4], st));
  // (mean and the lookup table are released in stream order when this scope ends)
  return PA_OK;
}

// all / any of a boolean column (GROUPBY_NUMERIC_AGG(all|any, bool), dataframe.cpp:1522-1524): bit-packed Arrow
// booleans from the min / max of the unpacked 0 / 1 bytes.  Appends to g->outs.
int run_bool_emit(pa_groupby* g, uint32_t extb) {
  cudaStream_t st = g->stream;
  const uint32_t G = g->G;
  const size_t words = (static_cast<size_t>(G) + 31) / 32 + 1;
  uint32_t* ptr[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
  int k = 0;
  for (uint32_t bit : {PA_AGG_BOOL_ALL, PA_AGG_BOOL_ANY}) {
    if (extb & bit) {
      g->outs.emplace_back();
      AggOut& o = g->outs.back();
      o.bit = bit;
      o.format = "b";
      o.width = 1;
      o.nullable = true;
      PA_TRY(o.values.alloc(words * 4, st));
      PA_TRY(o.valid.alloc(words * 4, st));
      ptr[k][0] = o.values.as<uint32_t>();
      ptr[k][1] = o.valid.as<uint32_t>();
    }
    ++k;
  }
  if (G > 0) {
    k_emit_bool<<<(G + 255) / 256, 256, 0, st>>>(g->res, G, ptr[0][0], ptr[0][1], ptr[1][0], ptr[1][1]);
    CUDA_TRY(cudaGetLastError());
    g->last_launches += 1;
    CUDA_TRY(cudaEventRecord(g->ev[4], st));
  }
  return PA_OK;
}

// all / any: the aggregates k_emit_bool reads (min / max of the 0 / 1 bytes, and the count)
uint32_t bool_helper_mask(uint32_t extb) {
  return extb ? (PA_AGG_COUNT | ((extb & PA_AGG_BOOL_ALL) ? PA_AGG_MIN : 0u) | ((extb & PA_AGG_BOOL_ANY) ? PA_AGG_MAX : 0u)) : 0u;
}

void keep_outputs(pa_groupby* g, uint32_t mask) {   // drops the outputs whose bit is not in `mask`
  g->outs.erase(std::remove_if(g->outs.begin(), g->outs.end(), [&](const AggOut& o) { return (o.bit & mask) == 0; }), g->outs.end());
}

// Aggregates the local pass, partial records (pa_merge_create, chunked) and the sharded step (records + distinct pairs) take
constexpr uint32_t LOCAL_AGGS = PA_AGG_ALL | PA_AGG_STAGE2 | PA_AGG_BOOL_ALL | PA_AGG_BOOL_ANY | PA_AGG_COUNT_DISTINCT;
constexpr uint32_t RECORD_AGGS = PA_AGG_ALL | PA_AGG_STAGE2 | PA_AGG_BOOL_ALL | PA_AGG_BOOL_ANY;
constexpr uint32_t SHARDED_AGGS = RECORD_AGGS | PA_AGG_COUNT_DISTINCT;

// Partial-record width (merge.cuh) of an aggregate set; `compact`: the sharded step's one-sector record
int record_words(uint32_t agg_mask, bool compact) {
  return compact ? REC_WORDS_COMPACT : ((agg_mask & PA_AGG_STAGE2) ? REC_WORDS_STAGE2 : REC_WORDS);
}

// count_distinct (distinct.cuh): ids + value bits -> two stable radix sorts -> boundary count.  Appends to g->outs.
int run_count_distinct(pa_groupby* g, const Column* val) {
  cudaStream_t st = g->stream;
  const uint32_t G = g->G;
  const int64_t n = g->n;
  if (n >= (1ll << 31)) return set_err(PA_ERR_INVALID, "count_distinct sorts with 32-bit positions: at most 2^31 - 1 rows");
  g->outs.emplace_back();
  AggOut& o = g->outs.back();
  o.bit = PA_AGG_COUNT_DISTINCT;
  o.format = "l";
  o.width = 8;
  o.nullable = false;
  PA_TRY(o.values.alloc(static_cast<size_t>(std::max<uint32_t>(G, 1)) * 8, st));
  if (G == 0) {
    g->cd_have = true;   // (no pairs)
    return PA_OK;
  }
  DevBuf distinct, id_a, id_b, bits_a, bits_b, tmp;
  PA_TRY(distinct.alloc(static_cast<size_t>(G) * 8, st));
  CUDA_TRY(cudaMemsetAsync(distinct.p, 0, static_cast<size_t>(G) * 8, st));
  if (n > 0) {
    RowLookup lk;
    PA_TRY(build_row_lookup(g, &lk));
    const size_t nn = static_cast<size_t>(n);
    PA_TRY(id_a.alloc(nn * 4, st));
    PA_TRY(id_b.alloc(nn * 4, st));
    PA_TRY(bits_a.alloc(nn * 8, st));
    PA_TRY(bits_b.alloc(nn * 8, st));
    DistinctFillArgs a{};
    a.ids = lk.a;
    a.vals = val->data;
    a.vvalid = val->valid;
    a.voff = val->bit_off;
    a.vw = val->width;
    a.out_bits = bits_a.as<uint64_t>();
    a.out_id = id_a.as<uint32_t>();
    const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, static_cast<int64_t>(g->num_sms) * 16)));
    if (val->vc == VC_F) k_distinct_fill<VC_F><<<grid, 256, 0, st>>>(a);
    else if (val->vc == VC_I) k_distinct_fill<VC_I><<<grid, 256, 0, st>>>(a);
    else k_distinct_fill<VC_U><<<grid, 256, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    // by value (64 bits; narrower columns need fewer), then stably by id (32 bits: kNoGroup must sort last)
    const int vbits = val->vc == VC_F ? 64 : (val->vc == VC_I ? 64 : std::min(64, val->width * 8));
    size_t t1 = 0, t2 = 0;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, t1, bits_a.as<uint64_t>(), bits_b.as<uint64_t>(), id_a.as<uint32_t>(), id_b.as<uint32_t>(),
                                             static_cast<int>(n), 0, vbits, st));
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, t2, id_b.as<uint32_t>(), id_a.as<uint32_t>(), bits_b.as<uint64_t>(), bits_a.as<uint64_t>(),
                                             static_cast<int>(n), 0, 32, st));
    PA_TRY(tmp.alloc(std::max(t1, t2), st));
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(tmp.p, t1, bits_a.as<uint64_t>(), bits_b.as<uint64_t>(), id_a.as<uint32_t>(), id_b.as<uint32_t>(),
                                             static_cast<int>(n), 0, vbits, st));
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(tmp.p, t2, id_b.as<uint32_t>(), id_a.as<uint32_t>(), bits_b.as<uint64_t>(), bits_a.as<uint64_t>(),
                                             static_cast<int>(n), 0, 32, st));
    const int64_t threads = (n + CD_PER_THREAD - 1) / CD_PER_THREAD;
    k_distinct_count<<<static_cast<int>((threads + 255) / 256), 256, 0, st>>>(id_a.as<uint32_t>(), bits_a.as<uint64_t>(), n, distinct.as<unsigned long long>());
    CUDA_TRY(cudaGetLastError());
    // the distinct pairs themselves, for the multi-GPU exchange: compacted into the sort's free buffers, then copied
    // to buffers of their own size (12 bytes per pair: at most half of the 24 bytes per row the sort needs)
    DevBuf cursor;
    PA_TRY(cursor.alloc(8, st));
    CUDA_TRY(cudaMemsetAsync(cursor.p, 0, 8, st));
    k_distinct_pairs<<<static_cast<int>((threads + 255) / 256), 256, 0, st>>>(id_a.as<uint32_t>(), bits_a.as<uint64_t>(), n, id_b.as<uint32_t>(),
                                                                           bits_b.as<uint64_t>(), cursor.as<unsigned long long>());
    CUDA_TRY(cudaGetLastError());
    unsigned long long d = 0;
    CUDA_TRY(cudaMemcpyAsync(&d, cursor.p, 8, cudaMemcpyDeviceToHost, st));
    id_a.reset(); bits_a.reset(); tmp.reset();
    CUDA_TRY(cudaStreamSynchronize(st));
    PA_TRY(g->cd_id.alloc(std::max<uint64_t>(d, 1) * 4, st));
    PA_TRY(g->cd_bits.alloc(std::max<uint64_t>(d, 1) * 8, st));
    if (d) {
      CUDA_TRY(cudaMemcpyAsync(g->cd_id.p, id_b.p, d * 4, cudaMemcpyDeviceToDevice, st));
      CUDA_TRY(cudaMemcpyAsync(g->cd_bits.p, bits_b.p, d * 8, cudaMemcpyDeviceToDevice, st));
    }
    g->cd_n = d;
  }
  g->cd_have = true;
  k_distinct_emit<<<(G + 255) / 256, 256, 0, st>>>(distinct.as<unsigned long long>(), G, o.values.as<int64_t>());
  CUDA_TRY(cudaGetLastError());
  g->last_launches += 6;
  CUDA_TRY(cudaEventRecord(g->ev[4], st));
  return PA_OK;
}

// ------------------------------ Arrow export ------------------------------
struct ExportPriv {
  void* bufs[3] = {nullptr, nullptr, nullptr};
  const void* ptrs[3] = {nullptr, nullptr, nullptr};
  std::string format;
};

void release_array(ArrowArray* a) {
  auto* p = static_cast<ExportPriv*>(a->private_data);
  if (p) {
    free(p->bufs[0]);
    free(p->bufs[1]);
    free(p->bufs[2]);
    delete p;
  }
  a->release = nullptr;
}
void release_schema(ArrowSchema* s) {
  delete static_cast<std::string*>(s->private_data);
  s->release = nullptr;
}

int export_host(cudaStream_t st, const std::string& format, int width, uint32_t G, const void* d_values,
                const uint32_t* d_valid, ArrowArray* out, ArrowSchema* out_schema) {
  auto* priv = new ExportPriv();
  const size_t vbytes = format == "b" ? (static_cast<size_t>(G) + 31) / 32 * 4 : static_cast<size_t>(G) * width;   // booleans are bit-packed
  priv->bufs[1] = malloc(std::max<size_t>(vbytes, 64));
  const size_t words = (static_cast<size_t>(G) + 31) / 32;
  int64_t null_count = 0;
  if (G > 0) {
    cudaError_t e = cudaMemcpyAsync(priv->bufs[1], d_values, vbytes, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && d_valid) {
      priv->bufs[0] = malloc(std::max<size_t>(words * 4, 64));
      e = cudaMemcpyAsync(priv->bufs[0], d_valid, words * 4, cudaMemcpyDeviceToHost, st);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
      free(priv->bufs[0]); free(priv->bufs[1]); delete priv;
      return set_err(PA_ERR_CUDA, "result copy failed: %s", cudaGetErrorString(e));
    }
    if (d_valid) {
      const uint32_t* w = static_cast<const uint32_t*>(priv->bufs[0]);
      int64_t set = 0;
      for (size_t i = 0; i < words; ++i) set += __builtin_popcount(w[i]);
      null_count = static_cast<int64_t>(G) - set;
      if (null_count == 0) { free(priv->bufs[0]); priv->bufs[0] = nullptr; }
    }
  }
  priv->ptrs[0] = priv->bufs[0];
  priv->ptrs[1] = priv->bufs[1];
  memset(out, 0, sizeof *out);
  out->length = G;
  out->null_count = null_count;
  out->offset = 0;
  out->n_buffers = 2;
  out->buffers = priv->ptrs;
  out->release = release_array;
  out->private_data = priv;
  memset(out_schema, 0, sizeof *out_schema);
  auto* f = new std::string(format);
  out_schema->format = f->c_str();
  out_schema->name = "";
  out_schema->flags = ARROW_FLAG_NULLABLE;
  out_schema->release = release_schema;
  out_schema->private_data = f;
  return PA_OK;
}

int ensure_device(pa_groupby* g) {
  CUDA_TRY(cudaSetDevice(g->device));
  return PA_OK;
}

int bits_for(uint64_t n_values) {  // bits needed to represent values 0..n_values-1
  int b = 1;
  while (b < 64 && (1ull << b) < n_values) ++b;
  return b;
}

// ---- composite keys: the packing layout (pa_key_layout) ----
static_assert(PA_MAX_KEY_COLS == kMaxKeyCols, "public key column limit");

// Value bits of a composite key's column: a dictionary column needs only enough for its codes
int key_bits(int width, bool is_dict, int64_t dict_len) {
  return (is_dict && dict_len > 0) ? bits_for(static_cast<uint64_t>(dict_len)) : width * 8;
}

// Bits a composite key packs into under layout l: value bits plus a null bit per nullable column
int layout_bits(const pa_key_layout& l) {
  int bits = 0;
  for (int j = 0; j < l.n_keys; ++j) bits += l.bits[j] + l.nullable[j];
  return bits;
}

// The one place the packing order is decided: column j at the bits after columns 0 .. j-1, value bits then null bit.
int layout_fields(const pa_key_layout& l, std::vector<KeyField>* fields) {
  const int total = layout_bits(l);
  if (total > 64) return set_err(PA_ERR_NOT_IMPLEMENTED, "composite key needs %d bits; only keys that pack into 64 bits are supported", total);
  fields->assign(l.n_keys, KeyField{});
  int shift = 0;
  for (int j = 0; j < l.n_keys; ++j) {
    KeyField& f = (*fields)[j];
    f.width = l.width[j]; f.bits = l.bits[j]; f.nullable = l.nullable[j];
    f.shift = shift;
    shift += f.bits + f.nullable;
  }
  return PA_OK;
}

// A layout from outside (caller, peer rank): `which` names it in the message
int check_layout(const pa_key_layout& l, int which) {
  if (l.n_keys < 2 || l.n_keys > PA_MAX_KEY_COLS)
    return set_err(PA_ERR_INVALID, "key layout %d: %d key columns (a composite key has 2 .. %d)", which, l.n_keys, PA_MAX_KEY_COLS);
  for (int j = 0; j < l.n_keys; ++j) {
    if ((l.width[j] != 4 && l.width[j] != 8) || l.bits[j] < 1 || l.bits[j] > l.width[j] * 8 || (l.nullable[j] != 0 && l.nullable[j] != 1))
      return set_err(PA_ERR_INVALID, "key layout %d, key column %d: width %d, bits %d, nullable %d is not a packable field", which, j,
                     l.width[j], l.bits[j], l.nullable[j]);
  }
  return PA_OK;
}

// The layout a local handle's key columns imply on their own: a null bit where the column has a validity bitmap
// (load_column keeps one only when null_count != 0).  Fingerprints stay 0 (fill_fingerprints).
void column_layout(const pa_groupby* g, pa_key_layout* l) {
  *l = pa_key_layout{};
  l->n_keys = static_cast<int32_t>(g->keys.size());
  for (int j = 0; j < l->n_keys; ++j) {
    const Column& k = g->keys[j];
    l->width[j] = k.width;
    l->bits[j] = key_bits(k.width, k.is_dict, k.dict_len);
    l->nullable[j] = k.valid != nullptr;
  }
}

// The layout the handle packs with now (its fields)
void fields_layout(const pa_groupby* g, pa_key_layout* l) {
  *l = pa_key_layout{};
  l->n_keys = static_cast<int32_t>(g->fields.size());
  for (int j = 0; j < l->n_keys; ++j) {
    l->width[j] = g->fields[j].width; l->bits[j] = g->fields[j].bits; l->nullable[j] = g->fields[j].nullable;
  }
}

// Bytes [off, off + bytes) of an Arrow buffer on the host (copied from the device when it lives there)
int host_bytes(const void* buf, size_t off, size_t bytes, bool on_dev, std::vector<uint8_t>* out) {
  out->resize(bytes);
  if (!bytes) return PA_OK;
  if (!buf) return set_err(PA_ERR_INVALID, "dictionary buffer is null");
  const char* p = static_cast<const char*>(buf) + off;
  if (on_dev) CUDA_TRY(cudaMemcpy(out->data(), p, bytes, cudaMemcpyDeviceToHost));
  else memcpy(out->data(), p, bytes);
  return PA_OK;
}

uint64_t fnv1a(uint64_t h, const void* p, size_t n) {
  const uint8_t* b = static_cast<const uint8_t*>(p);
  for (size_t i = 0; i < n; ++i) { h ^= b[i]; h *= 0x100000001B3ull; }
  return h;
}

// 64-bit hash of a dictionary's logical values: its format, its length, then for every entry its validity and (when
// valid) its bytes, length-prefixed for utf8 / binary.  Computed once per column; never 0 (0 = not a dictionary).
int dict_fingerprint(Column* k) {
  if (!k->is_dict || k->dict_fp) return PA_OK;
  const ArrowArray* d = k->dict;
  const ArrowSchema* s = k->dict_schema;
  if (!d || !s || !s->format) return set_err(PA_ERR_INVALID, "dictionary key column without its dictionary");
  const char* f = s->format;
  const bool var = (f[0] == 'u' || f[0] == 'U' || f[0] == 'z' || f[0] == 'Z') && f[1] == 0;
  const bool wide_off = f[0] == 'U' || f[0] == 'Z';
  int width = 0, vc = VC_I;
  if (!var) {
    if (f[0] == 'b') return set_err(PA_ERR_NOT_IMPLEMENTED, "dictionary of booleans in a composite key");
    PA_TRY(parse_format(f, &width, &vc));
  }
  if (d->n_buffers < (var ? 3 : 2)) return set_err(PA_ERR_INVALID, "dictionary of format '%s' has %lld buffers", f, (long long)d->n_buffers);
  const int64_t len = d->length, off = d->offset;
  std::vector<uint8_t> valid, vals, offs;
  const bool has_valid = d->null_count != 0 && d->buffers[0] != nullptr;
  if (has_valid) PA_TRY(host_bytes(d->buffers[0], static_cast<size_t>(off / 8), static_cast<size_t>((off + len + 7) / 8 - off / 8), k->dict_on_dev, &valid));
  int64_t first = 0;
  if (var) {
    const size_t ow = wide_off ? 8 : 4;
    PA_TRY(host_bytes(d->buffers[1], static_cast<size_t>(off) * ow, static_cast<size_t>(len + 1) * ow, k->dict_on_dev, &offs));
    auto at = [&](int64_t i) -> int64_t {
      if (wide_off) { int64_t v; memcpy(&v, offs.data() + i * 8, 8); return v; }
      int32_t v; memcpy(&v, offs.data() + i * 4, 4); return v;
    };
    first = at(0);
    const int64_t last = at(len);
    if (last < first) return set_err(PA_ERR_INVALID, "dictionary offsets are not ascending");
    PA_TRY(host_bytes(d->buffers[2], static_cast<size_t>(first), static_cast<size_t>(last - first), k->dict_on_dev, &vals));
    uint64_t h = fnv1a(0xCBF29CE484222325ull, f, strlen(f) + 1);
    h = fnv1a(h, &len, sizeof len);
    for (int64_t i = 0; i < len; ++i) {
      const uint8_t ok = has_valid ? ((valid[static_cast<size_t>((off % 8 + i) / 8)] >> ((off % 8 + i) % 8)) & 1) : 1;
      h = fnv1a(h, &ok, 1);
      if (!ok) continue;
      const int64_t b = at(i) - first, n = at(i + 1) - at(i);
      h = fnv1a(h, &n, sizeof n);
      h = fnv1a(h, vals.data() + b, static_cast<size_t>(n));
    }
    k->dict_fp = h ? h : 1;
    return PA_OK;
  }
  PA_TRY(host_bytes(d->buffers[1], static_cast<size_t>(off) * width, static_cast<size_t>(len) * width, k->dict_on_dev, &vals));
  uint64_t h = fnv1a(0xCBF29CE484222325ull, f, strlen(f) + 1);
  h = fnv1a(h, &len, sizeof len);
  for (int64_t i = 0; i < len; ++i) {
    const uint8_t ok = has_valid ? ((valid[static_cast<size_t>((off % 8 + i) / 8)] >> ((off % 8 + i) % 8)) & 1) : 1;
    h = fnv1a(h, &ok, 1);
    if (ok) h = fnv1a(h, vals.data() + i * width, static_cast<size_t>(width));
  }
  k->dict_fp = h ? h : 1;
  return PA_OK;
}

int fill_fingerprints(pa_groupby* g, pa_key_layout* l) {
  for (int j = 0; j < l->n_keys; ++j) {
    PA_TRY(dict_fingerprint(&g->keys[j]));
    l->dict_fingerprint[j] = g->keys[j].dict_fp;
  }
  return PA_OK;
}

// Packs the handle's key columns under g->fields into one 64-bit word per row
int pack_keys(pa_groupby* g) {
  const int nk = static_cast<int>(g->keys.size());
  KeyPackArgs a{};
  for (int j = 0; j < nk; ++j) {
    const Column& k = g->keys[j];
    const KeyField& f = g->fields[j];
    a.col[j] = k.data; a.valid[j] = k.valid; a.off[j] = k.bit_off; a.width[j] = k.width;
    a.bits[j] = f.bits; a.shift[j] = f.shift; a.nullable[j] = f.nullable;
  }
  PA_TRY(g->packed_keys.alloc(static_cast<size_t>(g->n) * 8, g->stream));
  a.n_cols = nk;
  a.n = g->n;
  a.out = g->packed_keys.as<uint64_t>();
  const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((g->n + 255) / 256, g->num_sms * 16)));
  k_pack_keys<<<grid, 256, 0, g->stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  g->packed = true;
  g->key_data = g->packed_keys.p;
  g->key_valid = nullptr;
  g->key_bit_off = 0;
  g->key_width = 8;
  return PA_OK;
}

// Collision hook for tests (PA_TEST_STR_HASH_BITS=b): hashes made under seed 0 keep only their low b bits, so that
// different keys share a hash on demand — utf8 keys and hashed composite keys alike.  Unset: every bit is kept.
uint64_t test_hash_keep(uint64_t seed) {
  static const char* bits = getenv("PA_TEST_STR_HASH_BITS");
  if (!bits || seed != 0) return ~0ull;
  const int b = atoi(bits);
  return b <= 0 ? 0ull : b >= 64 ? ~0ull : (1ull << b) - 1;
}

// A hashed key's words under g->key_seed: k_str_hash for one utf8 column (the words shards exchange), k_row_hash for a
// composite key
int hash_keys(pa_groupby* g) {
  cudaStream_t st = g->stream;
  const uint64_t seed = 0x5851F42D4C957F2Dull + g->key_seed * 0x9E3779B97F4A7C15ull, keep = test_hash_keep(g->key_seed);
  PA_TRY(g->packed_keys.alloc(static_cast<size_t>(std::max<int64_t>(g->n, 1)) * 8, st));
  uint64_t* out = g->packed_keys.as<uint64_t>();
  if (g->n > 0) {
    const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((g->n + 255) / 256, static_cast<int64_t>(g->num_sms) * 16)));
    const Column& k = g->keys[0];
    if (g->keys.size() == 1) k_str_hash<<<grid, 256, 0, st>>>(k.str, k.valid, k.bit_off, g->n, seed, keep, out);
    else k_row_hash<<<grid, 256, 0, st>>>(row_keys(g), seed, keep, out);
    CUDA_TRY(cudaGetLastError());
  }
  g->key_data = out;
  return PA_OK;
}

// Packed when the key is one fixed-width column (verbatim) or a composite key whose layout fits 64 bits (k_pack_keys);
// otherwise — a utf8 column, or more than 64 bits — hashed.
int setup_keys(pa_groupby* g) {
  const int nk = static_cast<int>(g->keys.size());
  if (nk > kMaxKeyCols) return set_err(PA_ERR_INVALID, "at most %d key columns", kMaxKeyCols);
  bool has_str = false;
  for (const Column& k : g->keys) {
    if (!k.is_str && k.width != 4 && k.width != 8) return set_err(PA_ERR_INVALID, "key columns must be 32- or 64-bit (format '%s')", k.format.c_str());
    has_str = has_str || k.is_str;
  }
  if (nk == 1) {
    const Column& k = g->keys[0];
    g->fields.assign(1, KeyField{});
    g->packed = false;
    g->key_data = k.data;
    g->key_valid = k.valid;
    g->key_bit_off = k.bit_off;
    g->key_width = k.width;
    g->fields[0].width = k.width;
    g->hashed = k.is_str;
    return k.is_str ? hash_keys(g) : PA_OK;
  }
  pa_key_layout own;
  column_layout(g, &own);
  if (!has_str && layout_bits(own) <= 64) {
    PA_TRY(layout_fields(own, &g->fields));
    return pack_keys(g);
  }
  g->fields.clear();
  g->packed = false;
  g->hashed = true;
  g->key_valid = nullptr;   // every row belongs to a regular group: nulls are part of the hashed row
  g->key_bit_off = 0;
  g->key_width = 8;
  return hash_keys(g);
}

// A merged handle's composite key: the records carry the packed word, pa_groupby_unique unpacks column j of it
int set_merged_layout(pa_groupby* g, const pa_key_layout& l, const char* const* key_formats) {
  std::vector<KeyField> fields;
  PA_TRY(layout_fields(l, &fields));
  std::vector<Column> keys(static_cast<size_t>(l.n_keys));
  for (int j = 0; j < l.n_keys; ++j) {
    if (!key_formats[j]) return set_err(PA_ERR_INVALID, "key_formats[%d] is null", j);
    int w = 8, vc = VC_I;
    PA_TRY(parse_format(key_formats[j], &w, &vc));
    if (w != l.width[j]) return set_err(PA_ERR_INVALID, "key_formats[%d] '%s' is %d bytes wide, the layout says %d", j, key_formats[j], w, l.width[j]);
    keys[j].format = key_formats[j];
    keys[j].width = w;
  }
  g->keys = std::move(keys);
  g->fields = std::move(fields);
  g->packed = true;
  return PA_OK;
}

// Drops everything computed from the handle's key words (after a repack or a rehash)
void drop_results(pa_groupby* g) {
  g->have_groups = false; g->bk_have_hist = false; g->G = 0; g->outs.clear();
  g->lk_valid = false;
  g->have_groupings = false;
  g->parts_n = 0;
  g->s2_ext = 0; g->s2_m2.reset(); g->s2_prod.reset();
  g->cd_have = false; g->cd_n = 0; g->cd_id.reset(); g->cd_bits.reset(); g->dp_parts_n = 0;
}

// Hashed key: rehash with hash seed `seed`; the next aggregate groups and checks anew
int set_key_seed(pa_groupby* g, uint64_t seed) {
  if (g->key_seed == seed) return PA_OK;
  g->key_seed = seed;
  PA_TRY(hash_keys(g));
  g->key_verified = false;
  drop_results(g);
  return PA_OK;
}

int aggregate_impl_raw(pa_groupby* g, const Column* val, uint32_t mask, bool deferred, int start_at);

// Hashed keys (one utf8 column, or a composite key that does not pack into 64 bits) are grouped by a seeded 64-bit
// hash; the first pass on a handle checks every row against its group's representative and, should two different
// keys ever share a hash, re-hashes with another seed and repeats (strkeys.cuh, rowkeys.cuh).
int aggregate_impl(pa_groupby* g, const Column* val, uint32_t mask, bool deferred = false, int start_at = 0) {
  if (!g->hashed || g->key_verified) return aggregate_impl_raw(g, val, mask, deferred, start_at);
  for (int attempt = 0; attempt < 4; ++attempt) {
    PA_TRY(aggregate_impl_raw(g, val, mask, false, attempt == 0 ? start_at : 0));
    bool collided = false;
    PA_TRY(verify_hashed_keys(g, &collided));
    if (!collided) { g->key_verified = true; return PA_OK; }
    PA_TRY(set_key_seed(g, g->key_seed + 1));
  }
  return set_err(PA_ERR_STATE, "%s: four differently seeded 64-bit hashes all collided", g->keys.size() == 1 ? "utf8 keys" : "hashed composite key");
}

int aggregate_impl_raw(pa_groupby* g, const Column* val, uint32_t mask, bool deferred, int start_at) {
  cudaStream_t st = g->stream;
  g->last_launches = 0;
  g->last_mode = 0; g->last_rlog = 0; g->last_passes = 0;
  g->unordered = false;
  const int vc = val ? val->vc : VC_I;
  const bool wide = is_wide(mask, vc);
  CUDA_TRY(cudaEventRecord(g->ev[0], st));
  if (g->resample) {
    CUDA_TRY(cudaEventRecord(g->ev[1], st));
    PA_TRY(run_resample(g, val, mask, wide));
    g->last_path = 3;
  } else {
    const int gmax = lc_gmax(vc, lc_is_wide(mask, vc));
    // (an earlier pass on this handle may already have told us how many groups there are)
    const int64_t known_groups = g->opt.expected_groups > 0 ? g->opt.expected_groups : (g->have_groups ? static_cast<int64_t>(g->G) : 0);
    bool try_low = g->opt.path != PA_PATH_GLOBAL && (known_groups <= gmax + 2 || g->opt.path == PA_PATH_LOWCARD);
    // the per-warp count words of the shared-memory path hold 24 bits next to the claim tag (lowcard.cuh): with
    // 148 SMs x >= 12 warps a warp sees at most 2^32 / 1776 = 2.4 M rows; a small MIG slice must not overflow them
    if (g->n / (static_cast<int64_t>(g->num_sms) * 12) >= (1ll << 24) - 1) try_low = false;
    bool done = false;
    if (start_at == 2) try_low = false;                       // (resuming after a deferred pass overflowed)
    // the groups of this handle's keys are known from an earlier dense pass: accumulate the sums only
    const bool known = try_low && start_at == 0 && !g->opt.lowcard_no_dense && lk_applies(g, val, mask);
    if (try_low && deferred && start_at == 0 && !g->opt.lowcard_no_dense) {
      // Deferred: queue the dense-mode pass and the emit without reading the status back.  If the pass turns
      // out to have declined / aborted / overflowed, finish_pending() resumes synchronously from there.
      LcOutcome oc = LC_DONE;
      if (known) PA_TRY(run_lowcard_known(g, val, mask, &oc, true));
      else PA_TRY(run_lowcard(g, val, mask, wide, false, &oc, true));
      g->last_path = PA_PATH_LOWCARD;
      g->have_groups = true;
      g->last_wide = wide;
      g->last_vc = vc;
      g->last_vw = val ? val->width : 8;
      g->last_vfmt = val ? val->format : "l";
      g->parts_n = 0;
      g->emit_G_dev = g->status.as<uint32_t>() + ST_NGROUPS;
      PA_TRY(run_emit(g, val, mask));
      g->emit_G_dev = nullptr;
      CUDA_TRY(cudaEventRecord(g->ev[4], st));
      g->pending = true;
      return PA_OK;
    }
    if (known) {
      LcOutcome oc = LC_DONE;
      PA_TRY(run_lowcard_known(g, val, mask, &oc, false));
      if (oc == LC_DONE) { done = true; try_low = false; g->last_path = PA_PATH_LOWCARD; }   // (else: the full pass below)
    }
    if (try_low) {
      LcOutcome oc = LC_DONE;
      PA_TRY(run_lowcard(g, val, mask, wide, g->opt.lowcard_no_dense != 0 || start_at == 1, &oc));
      if (oc == LC_DENSE_MISS) PA_TRY(run_lowcard(g, val, mask, wide, true, &oc));   // a key outside the sampled window
      if (oc == LC_DONE) { done = true; g->last_path = PA_PATH_LOWCARD; }
      else if (g->opt.path == PA_PATH_LOWCARD) return set_err(PA_ERR_INVALID, "more groups than the shared-memory path holds (%d)", gmax);
    }
    if (!done) {
      g->last_mode = 0; g->last_rlog = 0; g->last_passes += 1;
      PA_TRY(run_global(g, val, mask, wide));
      g->last_path = PA_PATH_GLOBAL;
    }
  }
  if (g->unordered) {   // sharded step: the records stay where the bucket aggregation left them; GroupResult, outputs
    CUDA_TRY(cudaEventRecord(g->ev[4], st));   // and group count of the handle are as before this pass
    return PA_OK;
  }
  g->have_groups = true;
  g->last_wide = wide;
  g->last_vc = vc;
  g->last_vw = val ? val->width : 8;
  g->last_vfmt = val ? val->format : "l";
  g->parts_n = 0;
  PA_TRY(run_emit(g, val, mask));
  CUDA_TRY(cudaEventRecord(g->ev[4], st));
  return PA_OK;
}

// ---- owner-side merge of partial records (merge.cuh) ----
int set_merged_formats(pa_groupby* g, const char* value_format, const char* key_format) {
  g->merged = true;
  g->packed = false;   // (pa_merge_set_key_layout makes it composite; a recycled handle may have been)
  g->keys.resize(1);
  int kw = 8, kvc = VC_I;
  // utf8 key: the records' key word is the hash; the strings come with pa_merge_key_strings
  g->ks_str = (key_format[0] == 'u' || key_format[0] == 'U') && key_format[1] == 0;
  g->ks_have = false;
  g->ks_off.reset(); g->ks_bytes.reset(); g->ks_rows.reset();
  if (!g->ks_str) PA_TRY(parse_format(key_format, &kw, &kvc));
  g->keys[0].format = key_format;
  g->keys[0].width = kw;
  g->fields.assign(1, KeyField{});
  g->fields[0].width = kw;
  g->index_format = key_format;
  PA_TRY(parse_format(value_format, &g->last_vw, &g->last_vc));
  g->last_vfmt = value_format;
  return PA_OK;
}

// GroupResult and fold outputs (64-bit counts, first / last values, global first rows) for `cap` groups, as outputs of `a`
template <typename Args>
int alloc_merged_result(pa_groupby* g, uint32_t cap, Args* a) {
  cudaStream_t st = g->stream;
  PA_TRY(alloc_result(g, cap, true, true));
  const size_t n = std::max<uint32_t>(cap, 1);
  PA_TRY(g->m_count64.alloc(n * 8, st));
  g->res.count64 = g->m_count64.as<uint64_t>();
  PA_TRY(g->m_first_val.alloc(n * 8, st));
  PA_TRY(g->m_first_row_g.alloc(n * 8, st));
  PA_TRY(g->m_last_val.alloc(n * 8, st));
  PA_TRY(g->m_first_valid.alloc(n, st));
  PA_TRY(g->m_last_valid.alloc(n, st));
  a->out = g->res;
  a->o_first_val = g->m_first_val.as<uint64_t>(); a->o_last_val = g->m_last_val.as<uint64_t>();
  a->o_first_valid = g->m_first_valid.as<uint8_t>(); a->o_last_valid = g->m_last_valid.as<uint8_t>();
  a->o_first_row_g = g->m_first_row_g.as<uint64_t>();
  return PA_OK;
}

// Scratch of one merge (key table, per-source index, compaction / sort buffers).  A communicator keeps one between
// steps (pa_groupby_sharded_aggregate) so that a step allocates nothing but its result.
struct MergeScratch { DevBuf tkeys, idx, m_first, m_slot, s_first, s_slot, cub_tmp; uint64_t last_slots = 0; };

// Common part of the merge entry points.  `d_off` = device array [n_sources + 1], exclusive prefix
// of the per-source record counts (the exact total is d_off[n_sources]); nrec_max = host-side upper bound.
int merge_build(pa_groupby* g, const void* dev_records, const uint64_t* d_off, int32_t n_sources, uint64_t nrec_max,
                uint32_t agg_mask, const char* value_format, const char* key_format, MergeScratch* keep = nullptr,
                uint64_t row_bound = 0, bool compact = false, uint64_t distinct_hint = 0) {
  cudaStream_t st = g->stream;
  PA_TRY(set_merged_formats(g, value_format, key_format));
  if (nrec_max >= 0xFFFFFFFFull) return set_err(PA_ERR_NOT_IMPLEMENTED, "more than 2^32-1 partial records per rank");
  MergeScratch local_scratch;
  MergeScratch& ms = keep ? *keep : local_scratch;
  DevBuf &tkeys = ms.tkeys, &idx = ms.idx, &m_first = ms.m_first, &m_slot = ms.m_slot, &s_first = ms.s_first, &s_slot = ms.s_slot, &cub_tmp = ms.cub_tmp;
  PA_TRY(m_first.alloc(std::max<uint64_t>(nrec_max, 1) * 8, st));
  PA_TRY(m_slot.alloc(std::max<uint64_t>(nrec_max, 1) * 4, st));
  MergeArgs a{};
  a.records = static_cast<const uint64_t*>(dev_records);
  a.src_offset = d_off;
  const uint32_t ext = agg_mask & PA_AGG_STAGE2;
  a.nsrc = n_sources; a.nrec = nrec_max;
  a.words = record_words(agg_mask, compact);
  a.status = g->status.as<uint32_t>();
  a.m_first_row = m_first.as<uint64_t>(); a.m_slot = m_slot.as<uint32_t>();
  a.vc = g->last_vc;
  // Join table: 2^k >= 2 x the number of distinct keys.  A source holds every key at most once, so the count lies
  // between the largest source and the sum; sources that saw (nearly) the same keys — row-range shards of one column —
  // are the common case, so the table is sized by `distinct_hint` (the largest source; 0 = unknown) first: 8 sources of
  // 12.5 M records fill 2^25 slots instead of 2^28 (index array 1 GB instead of 8.6 GB per step).  Too small shows as a
  // probe sequence beyond max_probe; then the merge is redone with the table every key set fits.
  uint32_t h_status[ST_WORDS];
  uint64_t sized_for = distinct_hint ? std::min<uint64_t>(std::max<uint64_t>(distinct_hint + distinct_hint / 4, 512), std::max<uint64_t>(nrec_max, 512)) : std::max<uint64_t>(nrec_max, 512);
  for (;;) {
    uint64_t cap = 1024;
    while (cap < sized_for * 2) cap <<= 1;
    const uint64_t nslots = cap + 2;
    ms.last_slots = nslots;
    PA_TRY(tkeys.alloc(nslots * 8, st));
    PA_TRY(idx.alloc(nslots * n_sources * 4, st));
    const int fgrid = static_cast<int>(std::min<uint64_t>((nslots + 255) / 256, static_cast<uint64_t>(g->num_sms) * 16));
    k_fill_u64<<<fgrid, 256, 0, st>>>(tkeys.as<unsigned long long>(), nslots, kEmptyKey);
    CUDA_TRY(cudaMemsetAsync(idx.p, 0xFF, nslots * n_sources * 4, st));
    a.tkeys = tkeys.as<unsigned long long>(); a.cap_mask = cap - 1; a.idx = idx.as<uint32_t>();
    a.max_probe = sized_for >= nrec_max ? cap : std::min<uint64_t>(cap, 2048);
    CUDA_TRY(cudaEventRecord(g->ev[1], st));
    if (nrec_max) {
      k_merge_insert<<<static_cast<int>((nrec_max + 255) / 256), 256, 0, st>>>(a);
      CUDA_TRY(cudaGetLastError());
    }
    k_merge_compact<<<static_cast<int>((nslots + MC_THREADS - 1) / MC_THREADS), MC_THREADS, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(g->ev[2], st));
    CUDA_TRY(cudaMemcpyAsync(h_status, g->status.p, sizeof h_status, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (h_status[ST_PEER_OVERFLOW]) return set_err(PA_ERR_STATE, "a source rank had more groups than a padded block holds; use the counted exchange");
    if (h_status[ST_OVERFLOW] && sized_for < nrec_max) {   // the hint was too small: every key set fits a table sized by the record count
      sized_for = nrec_max;
      CUDA_TRY(cudaMemsetAsync(a.status + ST_OVERFLOW, 0, sizeof(uint32_t), st));
      CUDA_TRY(cudaMemsetAsync(a.status + ST_COUNTER, 0, sizeof(uint32_t), st));
      continue;
    }
    if (h_status[ST_OVERFLOW]) return set_err(PA_ERR_CUDA, "merge table overflow");
    break;
  }
  const uint32_t G = h_status[ST_COUNTER];
  g->G = G;
  // all / any: folded as min / max of the 0 / 1 bytes and the count, which is what k_emit_bool reads
  const uint32_t extb = agg_mask & (PA_AGG_BOOL_ALL | PA_AGG_BOOL_ANY);
  const uint32_t fold_mask = (agg_mask & (PA_AGG_ALL | PA_AGG_STAGE2)) | bool_helper_mask(extb);
  const bool wide = is_wide(fold_mask, g->last_vc);
  g->last_wide = wide;
  PA_TRY(alloc_merged_result(g, G, &a));
  if (ext & (AGG_VARIANCE | AGG_STDDEV)) PA_TRY(g->s2_m2.alloc(static_cast<size_t>(std::max<uint32_t>(G, 1)) * 8, st));
  if (ext & AGG_PRODUCT) PA_TRY(g->s2_prod.alloc(static_cast<size_t>(std::max<uint32_t>(G, 1)) * 8, st));
  uint32_t h_no_terms = 0;
  if (G) {
    PA_TRY(s_first.alloc(static_cast<size_t>(G) * 8, st));
    PA_TRY(s_slot.alloc(static_cast<size_t>(G) * 4, st));
    size_t tmp_bytes = 0;
    // (global first rows are below row_bound when the caller knows the shards: sort only the bits that can differ)
    int end_bit = 64;
    if (row_bound) { end_bit = 1; while (end_bit < 64 && (row_bound >> end_bit)) ++end_bit; }
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, m_first.as<uint64_t>(), s_first.as<uint64_t>(), m_slot.as<uint32_t>(), s_slot.as<uint32_t>(), static_cast<int>(G), 0, end_bit, st));
    PA_TRY(cub_tmp.alloc(tmp_bytes, st));
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(cub_tmp.p, tmp_bytes, m_first.as<uint64_t>(), s_first.as<uint64_t>(), m_slot.as<uint32_t>(), s_slot.as<uint32_t>(), static_cast<int>(G), 0, end_bit, st));
    a.order = s_slot.as<uint32_t>();
    a.G = G;
    if (ext) {
      a.o_m2 = (ext & (AGG_VARIANCE | AGG_STDDEV)) ? g->s2_m2.as<double>() : nullptr;
      a.o_prod = (ext & AGG_PRODUCT) ? g->s2_prod.as<unsigned long long>() : nullptr;
      k_merge_fold<true><<<(G + 255) / 256, 256, 0, st>>>(a);
      CUDA_TRY(cudaGetLastError());
      CUDA_TRY(cudaMemcpyAsync(&h_no_terms, a.status + ST_NO_TERMS, sizeof h_no_terms, cudaMemcpyDeviceToHost, st));
    } else {
      k_merge_fold<false><<<(G + 255) / 256, 256, 0, st>>>(a);
      CUDA_TRY(cudaGetLastError());
    }
  }
  CUDA_TRY(cudaEventRecord(g->ev[3], st));
  g->have_groups = true;
  g->last_launches = 4;
  g->last_path = 4;
  PA_TRY(run_emit(g, nullptr, fold_mask));
  if (ext) {
    PA_TRY(emit_stage2(g, g->last_vc, ext));
    g->last_launches += 1;
  }
  if (extb) {
    // (the helper min / max / count outputs are bytes and counts nobody asked for)
    keep_outputs(g, agg_mask);
    PA_TRY(run_bool_emit(g, extb));
  }
  CUDA_TRY(cudaEventRecord(g->ev[4], st));
  CUDA_TRY(cudaStreamSynchronize(st));   // local scratch (table, idx, sort buffers) is released after this point
  if (h_no_terms) return set_err(PA_ERR_STATE, "partial records carry no variance / product terms for this aggregate mask "
                                               "(export them with pa_groupby_partials_export_stage2 after an aggregate that computes them)");
  return PA_OK;
}

// Merge of records whose per-source counts the host knows: offsets to the device, the table sized by the largest source.
int merge_counted(pa_groupby* g, const void* dev_records, const int64_t* counts, int32_t n_sources, uint32_t agg_mask,
                  const char* value_format, const char* key_format, MergeScratch* keep, uint64_t row_bound, bool compact) {
  cudaStream_t st = g->stream;
  std::vector<uint64_t> off(n_sources + 1, 0);
  for (int i = 0; i < n_sources; ++i) off[i + 1] = off[i] + static_cast<uint64_t>(counts[i]);
  if (off[n_sources] && !dev_records) return set_err(PA_ERR_INVALID, "null record buffer");
  DevBuf d_off;
  PA_TRY(d_off.alloc(sizeof(uint64_t) * (n_sources + 1), st));
  CUDA_TRY(cudaMemcpyAsync(d_off.p, off.data(), sizeof(uint64_t) * (n_sources + 1), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemsetAsync(g->status.p, 0, sizeof(uint32_t) * ST_WORDS, st));
  CUDA_TRY(cudaEventRecord(g->ev[0], st));
  return merge_build(g, dev_records, d_off.as<uint64_t>(), n_sources, off[n_sources], agg_mask, value_format, key_format, keep,
                     row_bound, compact, static_cast<uint64_t>(*std::max_element(counts, counts + n_sources)));
}

int merge_padded_general(pa_groupby* g, const void* dev_blocks, int32_t n_sources, int64_t block_records, uint32_t agg_mask,
                         const char* value_format, const char* key_format) {
  cudaStream_t st = g->stream;
  const uint64_t nrec_max = static_cast<uint64_t>(n_sources) * static_cast<uint64_t>(block_records);
  DevBuf d_off, records;
  PA_TRY(d_off.alloc(sizeof(uint64_t) * (n_sources + 1), st));
  PA_TRY(records.alloc(nrec_max * PA_PARTIAL_WORDS * 8, st));
  CUDA_TRY(cudaMemsetAsync(g->status.p, 0, sizeof(uint32_t) * ST_WORDS, st));
  k_merge_unpad<<<n_sources, 256, 0, st>>>(static_cast<const uint64_t*>(dev_blocks), static_cast<uint32_t>(n_sources),
                                           static_cast<uint64_t>(block_records), records.as<uint64_t>(), d_off.as<uint64_t>(),
                                           g->status.as<uint32_t>());
  CUDA_TRY(cudaGetLastError());
  return merge_build(g, records.p, d_off.as<uint64_t>(), n_sources, nrec_max, agg_mask, value_format, key_format);
}

// Completes a deferred aggregate: reads the status words; on success only the group count was missing, otherwise
// the pass is redone synchronously from the stage that failed.
int finish_pending(pa_groupby* g) {
  if (g->pending_merge) {
    g->pending_merge = false;
    cudaStream_t st = g->stream;
    CUDA_TRY(cudaSetDevice(g->device));
    uint32_t h_status[ST_WORDS];
    CUDA_TRY(cudaMemcpyAsync(h_status, g->status.p, sizeof h_status, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (h_status[ST_PEER_OVERFLOW]) {
      g->have_groups = false; g->G = 0; g->outs.clear(); g->poolable = false;
      return set_err(PA_ERR_STATE, "a source rank had more groups than a padded block holds; use the counted exchange");
    }
    if (!h_status[ST_OVERFLOW]) {
      g->G = h_status[ST_COUNTER];
      return PA_OK;
    }
    g->outs.clear();                                    // too many records / groups for one CTA: general merge
    g->have_groups = false;
    g->poolable = false;
    if (!g->packed)
      return merge_padded_general(g, g->pm_blocks, g->pm_nsrc, g->pm_block_records, g->pm_mask, g->pm_vfmt.c_str(), g->pm_kfmt.c_str());
    // composite key (pa_merge_set_key_layout): the general merge sets the key format anew, the layout stays
    pa_key_layout l;
    fields_layout(g, &l);
    std::vector<std::string> kf;
    for (const Column& k : g->keys) kf.push_back(k.format);
    PA_TRY(merge_padded_general(g, g->pm_blocks, g->pm_nsrc, g->pm_block_records, g->pm_mask, g->pm_vfmt.c_str(), g->pm_kfmt.c_str()));
    std::vector<const char*> kp;
    for (const std::string& s : kf) kp.push_back(s.c_str());
    return set_merged_layout(g, l, kp.data());
  }
  if (!g->pending) return PA_OK;
  g->pending = false;
  cudaStream_t st = g->stream;
  CUDA_TRY(cudaSetDevice(g->device));
  uint32_t h_status[ST_WORDS];
  CUDA_TRY(cudaMemcpyAsync(h_status, g->status.p, sizeof h_status, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  const Column* val = g->pending_has_val ? &g->pending_val : nullptr;
  int rc = PA_OK;
  const bool recorded = g->pending_lk_record;
  g->pending_lk_record = false;
  if (!h_status[ST_OVERFLOW] && !h_status[ST_DENSE_MISS]) {
    g->G = h_status[ST_NGROUPS];
    g->last_mode = static_cast<int>(h_status[ST_MODE]);
    g->last_rlog = static_cast<int>(h_status[ST_RLOG]);
    g->last_passes = 1;
    if (recorded && h_status[ST_MODE] == 1u && !(g->pending_had_groups && g->pending_prev_G != g->G)) g->lk_valid = true;
  } else {
    const int passes = h_status[ST_DENSE_MISS] == 2u ? 0 : 1;
    // a sum-only pass that met keys its facts do not describe drops them and redoes the full dense pass
    const bool known = h_status[ST_MODE] == LK_MODE;
    g->lk_valid = false;
    g->have_groups = g->pending_had_groups;
    g->G = g->pending_prev_G;
    rc = aggregate_impl(g, val, g->pending_mask, false, known ? 0 : (h_status[ST_OVERFLOW] ? 2 : 1));
    g->last_passes += passes;
  }
  if (rc == PA_OK && g->pending_had_groups && g->pending_prev_G != g->G)
    rc = set_err(PA_ERR_STATE, "group count changed between passes (%u vs %u)", g->pending_prev_G, g->G);
  return rc;
}

}  // namespace

namespace {

template <int VC, bool WIDE>
int run_resample_t(pa_groupby* g, const Column* val, uint32_t mask) {
  using SlotT = typename SlotOf<WIDE>::type;
  cudaStream_t st = g->stream;
  const int64_t nbins = g->rs.nbins;
  const uint64_t nslots = static_cast<uint64_t>(nbins) + 2;
  DevBuf &table = g->scr.table, &bnd = g->scr.bnd;
  PA_TRY(table.alloc(nslots * sizeof(SlotT), st));
  CUDA_TRY(cudaMemsetAsync(g->status.p, 0, sizeof(uint32_t) * ST_WORDS, st));
  const int init_grid = static_cast<int>(std::min<uint64_t>((nslots + 255) / 256, static_cast<uint64_t>(g->num_sms) * 16));
  k_gtable_init<WIDE><<<init_grid, 256, 0, st>>>(table.as<SlotT>(), nslots);
  CUDA_TRY(cudaGetLastError());
  const int64_t chunk = rs_chunk_rows(g->n);
  const int64_t nchunks = (g->n + chunk - 1) / chunk;
  PA_TRY(bnd.alloc(static_cast<size_t>(std::max<int64_t>(nchunks, 1)) * 2 * sizeof(RsPartial), st));
  if (nchunks > 0) {
    k_rs_init_bnd<<<static_cast<int>((nchunks * 2 + 255) / 256), 256, 0, st>>>(bnd.as<RsPartial>(), nchunks * 2);
    CUDA_TRY(cudaGetLastError());
  }
  RsArgs a{};
  a.ts = static_cast<const int64_t*>(g->key_data);
  a.vals = val ? val->data : nullptr;
  a.vvalid = val ? val->valid : nullptr;
  a.voff = val ? val->bit_off : 0;
  a.vw = val ? val->width : 8;
  a.n = g->n;
  a.spec = g->rs;
  a.table = table.p;
  a.bnd = bnd.as<RsPartial>();
  a.nchunks = nchunks;
  a.chunk = chunk;
  a.status = g->status.as<uint32_t>();
  a.agg_mask = mask;
  if (nchunks > 0) {
    const int64_t warps_per_block = RS_THREADS / 32;
    int per_sm = 1;   // one full wave of resident CTAs: the kernel is a grid-stride loop over chunks
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_resample_scan<VC, WIDE>, RS_THREADS, 0));
    const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((nchunks + warps_per_block - 1) / warps_per_block,
                                                                           static_cast<int64_t>(g->num_sms) * std::max(per_sm, 1))));
    k_resample_scan<VC, WIDE><<<grid, RS_THREADS, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(g->ev[2], st));
    k_resample_fixup<VC, WIDE><<<static_cast<int>((nchunks * 2 + 255) / 256), 256, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    g->last_launches += 4;
  } else {
    CUDA_TRY(cudaEventRecord(g->ev[2], st));
  }
  // occupied buckets -> first-appearance (= time) order -> GroupResult
  const uint64_t max_groups = std::min<uint64_t>(nslots, static_cast<uint64_t>(g->n) + 2);
  DevBuf &c_first = g->scr.c_first, &c_slot = g->scr.c_slot, &s_slot = g->scr.s_slot;
  PA_TRY(c_first.alloc(max_groups * 4, st));
  PA_TRY(c_slot.alloc(max_groups * 4, st));
  const int cgrid = static_cast<int>(std::min<uint64_t>((nslots + 255) / 256, static_cast<uint64_t>(g->num_sms) * 16));
  k_gtable_compact<WIDE><<<cgrid, 256, 0, st>>>(table.as<SlotT>(), nslots, c_first.as<uint32_t>(), c_slot.as<uint32_t>(), g->status.as<uint32_t>());
  CUDA_TRY(cudaGetLastError());
  g->last_launches += 1;
  uint32_t h_status[ST_WORDS];
  CUDA_TRY(cudaMemcpyAsync(h_status, g->status.p, sizeof h_status, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  if (h_status[ST_UNSORTED]) return set_err(PA_ERR_INVALID, "resample: the index must be sorted ascending (Values falls before first bin / after last bin)");
  const uint32_t G = h_status[ST_COUNTER];
  g->G = G;
  PA_TRY(alloc_result(g, G, WIDE, VC != VC_F));
  if (G > 0) {
    PA_TRY(s_slot.alloc(static_cast<size_t>(G) * 4, st));
    PA_TRY(order_by_first_row(g, c_first.as<uint32_t>(), c_slot.as<uint32_t>(), G, s_slot.as<uint32_t>()));
    k_gtable_gather<WIDE><<<(G + 255) / 256, 256, 0, st>>>(table.as<SlotT>(), static_cast<uint64_t>(nbins), s_slot.as<uint32_t>(), G, g->res);
    CUDA_TRY(cudaGetLastError());
    g->last_launches += 1;
  }
  CUDA_TRY(cudaEventRecord(g->ev[3], st));
  return PA_OK;
}

int run_resample(pa_groupby* g, const Column* val, uint32_t mask, bool wide) {
  const int vc = val ? val->vc : VC_I;
  if (val && val->vc == VC_F && val->width != 4 && val->width != 8) return set_err(PA_ERR_INVALID, "bad float width");
  if (wide) {
    if (vc == VC_F) return run_resample_t<VC_F, true>(g, val, mask);
    if (vc == VC_I) return run_resample_t<VC_I, true>(g, val, mask);
    return run_resample_t<VC_U, true>(g, val, mask);
  }
  if (vc == VC_F) return run_resample_t<VC_F, false>(g, val, mask);
  if (vc == VC_I) return run_resample_t<VC_I, false>(g, val, mask);
  return run_resample_t<VC_U, false>(g, val, mask);
}

int64_t floor_div(int64_t a, int64_t b) {
  int64_t q = a / b;
  if ((a % b != 0) && ((a < 0) != (b < 0))) --q;
  return q;
}

// adjustDatesAnchored (/root/reference/src/resample.cpp:85-178) on integer ticks; tz is not supported.
void anchor_range(int64_t start, int64_t end, int64_t freq, bool closed_right, int origin, int64_t origin_custom,
                  int64_t offset, int64_t ticks_per_day, int64_t* first, int64_t* last) {
  int64_t f = start, l = end, o = 0;
  switch (origin) {
    case 1: o = f; break;                                            // Start
    case 2: o = floor_div(f, ticks_per_day) * ticks_per_day; break;  // StartDay (default)
    case 3: o = l; break;                                            // End
    case 4: o = floor_div(l, ticks_per_day) * ticks_per_day; break;  // EndDay
    case 5: o = origin_custom; break;                                // Custom
    default: o = 0;                                                  // Epoch
  }
  o += offset;
  const int64_t fo = (f - o) % freq, lo = (l - o) % freq;            // truncating %, like the reference
  if (closed_right) {
    f -= (fo > 0) ? fo : freq;
    if (lo > 0) l += freq - lo;
  } else {
    if (fo > 0) f -= fo;
    l += (lo > 0) ? freq - lo : freq;
  }
  *first = f;
  *last = l;
}

}  // namespace

extern "C" {

const char* pa_last_error(void) { return g_err.c_str(); }
int pa_version(void) { return 100; }

void pa_options_init(pa_options* opt) {
  memset(opt, 0, sizeof *opt);
  opt->device = -1;
  opt->path = PA_PATH_AUTO;
}

int pa_device_count(int* out) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) { *out = 0; return set_err(PA_ERR_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e)); }
  *out = n;
  return PA_OK;
}

// Merged (multi-GPU) handles are created and destroyed once per step; their events, status buffer and
// result buffers are recycled through a small pool instead of being re-created (≈ 0.2 ms per step).
static std::mutex g_pool_mutex;
static std::vector<pa_groupby*> g_merge_pool;

static pa_groupby* pool_take(int device, cudaStream_t stream) {
  std::lock_guard<std::mutex> lock(g_pool_mutex);
  for (size_t i = 0; i < g_merge_pool.size(); ++i) {
    pa_groupby* h = g_merge_pool[i];
    if (h->device == device && h->stream == stream) {
      g_merge_pool.erase(g_merge_pool.begin() + i);
      return h;
    }
  }
  return nullptr;
}

static int handle_init(pa_groupby* g, const pa_options* opt) {
  if (opt) g->opt = *opt; else pa_options_init(&g->opt);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return set_err(PA_ERR_CUDA, "no CUDA device: pandasarrow_b200 has no CPU fallback");
  if (g->opt.device < 0) CUDA_TRY(cudaGetDevice(&g->device)); else g->device = g->opt.device;
  CUDA_TRY(cudaSetDevice(g->device));
  CUDA_TRY(cudaDeviceGetAttribute(&g->num_sms, cudaDevAttrMultiProcessorCount, g->device));
  if (g->opt.cuda_stream) { g->stream = static_cast<cudaStream_t>(g->opt.cuda_stream); g->own_stream = false; }
  else { CUDA_TRY(cudaStreamCreate(&g->stream)); g->own_stream = true; }
  cudaMemPool_t pool;
  CUDA_TRY(cudaDeviceGetDefaultMemPool(&pool, g->device));
  uint64_t keep = UINT64_MAX;
  CUDA_TRY(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
  for (auto& e : g->ev) CUDA_TRY(cudaEventCreate(&e));
  PA_TRY(g->status.alloc(sizeof(uint32_t) * ST_WORDS, g->stream));
  return PA_OK;
}

struct HandleDeleter {
  void operator()(pa_groupby* g) const { pa_groupby_destroy(g); }
};
using HandlePtr = std::unique_ptr<pa_groupby, HandleDeleter>;

int pa_groupby_create(const struct ArrowDeviceArray* keys, const struct ArrowSchema* key_schemas, int32_t n_keys,
                      const pa_options* opt, pa_groupby** out) {
  if (!keys || !key_schemas || n_keys < 1 || !out) return set_err(PA_ERR_INVALID, "pa_groupby_create: null argument");
  HandlePtr g(new pa_groupby());
  PA_TRY(handle_init(g.get(), opt));
  g->keys.resize(n_keys);
  for (int i = 0; i < n_keys; ++i) {
    const char* kf = key_schemas[i].format;
    if (kf && (kf[0] == 'u' || kf[0] == 'U') && kf[1] == 0) {
      PA_TRY(load_string_key(&keys[i], &key_schemas[i], g->stream, g->device, &g->keys[i]));
    } else {
      PA_TRY(load_column(&keys[i], &key_schemas[i], g->stream, g->device, &g->keys[i]));
    }
    if (g->keys[i].n != g->keys[0].n) return set_err(PA_ERR_INVALID, "key columns differ in length");
  }
  g->n = g->keys[0].n;
  if (g->n >= 0xFFFFFFFEll) return set_err(PA_ERR_NOT_IMPLEMENTED, "more than 2^32-2 rows per call; shard by row range");
  PA_TRY(setup_keys(g.get()));
  *out = g.release();
  return PA_OK;
}

static int ensure_groups(pa_groupby* g) {
  PA_TRY(finish_pending(g));
  if (g->have_groups) return PA_OK;
  PA_TRY(ensure_device(g));
  return aggregate_impl(g, nullptr, 0);
}

int pa_groupby_num_groups(pa_groupby* g, int64_t* out) {
  if (!g || !out) return set_err(PA_ERR_INVALID, "null argument");
  PA_TRY(ensure_groups(g));
  *out = g->G;
  return PA_OK;
}

static int unique_strings(pa_groupby* g, const StrCol& col, const uint32_t* rows, const uint8_t* kind, bool large, struct ArrowArray* out,
                          struct ArrowSchema* out_schema);

// unique(j) of a hashed key: column j at every group's first row, with its validity
static int unique_hashed(pa_groupby* g, int32_t key_i, struct ArrowArray* out, struct ArrowSchema* out_schema) {
  cudaStream_t st = g->stream;
  const Column& k = g->keys[key_i];
  const uint32_t G = g->G;
  DevBuf kind, vals, valid;
  PA_TRY(kind.alloc(std::max<uint32_t>(G, 1), st));
  if (!k.is_str) PA_TRY(vals.alloc(static_cast<size_t>(std::max<uint32_t>(G, 1)) * k.width, st));
  if (G) {
    k_gather_rep<<<(G + 255) / 256, 256, 0, st>>>(k.is_str ? nullptr : k.data, k.width, k.valid, k.bit_off, g->res.first_row, G, vals.p, kind.as<uint8_t>());
    CUDA_TRY(cudaGetLastError());
  }
  if (k.is_str) return unique_strings(g, k.str, g->res.first_row, kind.as<uint8_t>(), k.str.wide != 0, out, out_schema);
  PA_TRY(valid.alloc(((static_cast<size_t>(G) + 31) / 32 + 1) * 4, st));
  if (G) {
    k_kind_validity<<<(G + 31) / 32 * 32 / 256 + 1, 256, 0, st>>>(kind.as<uint8_t>(), G, valid.as<uint32_t>());
    CUDA_TRY(cudaGetLastError());
  }
  return export_host(st, k.format, k.width, G, vals.p, valid.as<uint32_t>(), out, out_schema);
}

int pa_groupby_unique(pa_groupby* g, int32_t key_i, struct ArrowArray* out, struct ArrowSchema* out_schema) {
  if (!g || !out || !out_schema) return set_err(PA_ERR_INVALID, "null argument");
  PA_TRY(ensure_groups(g));
  PA_TRY(ensure_device(g));
  if (g->hashed) {
    if (key_i < 0 || key_i >= static_cast<int>(g->keys.size())) return set_err(PA_ERR_INVALID, "key index %d out of range", key_i);
    if (g->keys.size() == 1) return unique_strings(g, g->keys[0].str, g->res.first_row, g->res.key_kind, g->keys[0].str.wide != 0, out, out_schema);
    return unique_hashed(g, key_i, out, out_schema);
  }
  if (g->merged && g->ks_str) {
    if (key_i != 0) return set_err(PA_ERR_INVALID, "key index %d out of range", key_i);
    if (!g->ks_have) return set_err(PA_ERR_STATE, "utf8 merged handle without its key strings: call pa_merge_key_strings first");
    const StrCol col{g->ks_off.p, g->ks_bytes.as<uint8_t>(), 1};
    return unique_strings(g, col, g->ks_rows.as<uint32_t>(), g->res.key_kind, g->keys[0].format == "U", out, out_schema);
  }
  if (g->resample) {
    if (key_i != 0) return set_err(PA_ERR_INVALID, "key index %d out of range", key_i);
    return export_host(g->stream, g->index_format, 8, g->G, g->res.key, nullptr, out, out_schema);
  }
  if (key_i < 0 || key_i >= static_cast<int>(g->keys.size())) return set_err(PA_ERR_INVALID, "key index %d out of range", key_i);
  const KeyField& f = g->fields[key_i];
  const uint32_t G = g->G;
  DevBuf vals, valid;
  PA_TRY(vals.alloc(static_cast<size_t>(std::max<uint32_t>(G, 1)) * f.width, g->stream));
  PA_TRY(valid.alloc(((static_cast<size_t>(G) + 31) / 32 + 1) * 4, g->stream));
  if (G > 0) {
    KeyEmitArgs a{};
    a.key = g->res.key; a.key_kind = g->res.key_kind; a.G = G;
    a.width = f.width; a.bits = f.bits; a.shift = f.shift; a.nullable = f.nullable; a.packed = g->packed;
    a.out = vals.p; a.out_valid = valid.as<uint32_t>();
    k_emit_key<<<(G + 255) / 256, 256, 0, g->stream>>>(a);
    CUDA_TRY(cudaGetLastError());
  }
  return export_host(g->stream, g->keys[key_i].format, f.width, G, vals.p, valid.as<uint32_t>(), out, out_schema);
}

static int aggregate_entry(pa_groupby* g, const struct ArrowDeviceArray* values, const struct ArrowSchema* value_schema,
                           uint32_t agg_mask, bool deferred) {
  if (!g || !values || !value_schema) return set_err(PA_ERR_INVALID, "null argument");
  if (agg_mask == 0 || (agg_mask & ~LOCAL_AGGS)) return set_err(PA_ERR_INVALID, "bad aggregate mask 0x%x", agg_mask);
  const uint32_t requested = agg_mask;
  const uint32_t extb = agg_mask & (PA_AGG_BOOL_ALL | PA_AGG_BOOL_ANY);
  const bool want_distinct = (agg_mask & PA_AGG_COUNT_DISTINCT) != 0;
  if (want_distinct && g->merged) return set_err(PA_ERR_NOT_IMPLEMENTED, "count_distinct is not available on merged (multi-GPU) handles");
  // product / variance / stddev: a second pass after the ordinary one, which then has to deliver count (and the mean)
  const uint32_t ext = agg_mask & PA_AGG_STAGE2;
  if (ext && g->merged) return set_err(PA_ERR_NOT_IMPLEMENTED, "product / variance / stddev are not available on merged (multi-GPU) handles");
  if (extb && g->merged) return set_err(PA_ERR_NOT_IMPLEMENTED, "all / any are not available on merged (multi-GPU) handles");
  if (ext || extb || want_distinct) {
    deferred = false;
    // all = (min over the 0 / 1 bytes) != 0, any = (max) != 0: the ordinary pass delivers both
    agg_mask = (agg_mask & PA_AGG_ALL) | PA_AGG_COUNT | ((ext & (PA_AGG_VARIANCE | PA_AGG_STDDEV)) ? PA_AGG_MEAN : 0u) | bool_helper_mask(extb);
  }
  PA_TRY(ensure_device(g));
  Column val;
  PA_TRY(load_column(values, value_schema, g->stream, g->device, &val));
  if (val.n != g->n) return set_err(PA_ERR_INVALID, "value column has %lld rows, keys have %lld", (long long)val.n, (long long)g->n);
  if (value_schema->dictionary) return set_err(PA_ERR_INVALID, "dictionary-encoded value columns are not aggregatable");
  if (val.is_bool && (requested & ~(PA_AGG_COUNT | PA_AGG_BOOL_ALL | PA_AGG_BOOL_ANY | PA_AGG_COUNT_DISTINCT)))
    return set_err(PA_ERR_INVALID, "boolean columns aggregate with count / all / any only");
  if (extb && !val.is_bool) return set_err(PA_ERR_INVALID, "all / any need a boolean column (arrow::compute has no kernel for other types)");
  uint32_t prev_G = g->G;
  bool had = g->have_groups;
  if (g->pending && deferred && !val.own_data.p && !val.own_valid.p) {
    // A deferred pass whose results nobody asked for is superseded by this one (its buffers are recycled in
    // stream order); had it failed, this pass fails the same way and is redone when it is finished.
    g->pending = false;
    prev_G = g->pending_prev_G;
    had = g->pending_had_groups;
    g->have_groups = had;
    g->G = prev_G;
  } else {
    PA_TRY(finish_pending(g));
    prev_G = g->G;
    had = g->have_groups;
  }
  // deferred mode needs inputs that outlive the call: device-resident columns only
  deferred = deferred && !val.own_data.p && !val.own_valid.p && !g->resample && !g->merged;
  if (deferred) {
    g->pending_val = Column{};
    g->pending_val.data = val.data; g->pending_val.valid = val.valid; g->pending_val.bit_off = val.bit_off;
    g->pending_val.n = val.n; g->pending_val.width = val.width; g->pending_val.vc = val.vc; g->pending_val.format = val.format;
    g->pending_has_val = true;
    g->pending_mask = agg_mask;
    g->pending_prev_G = prev_G;
    g->pending_had_groups = had;
  }
  // the stage-2 terms of an earlier aggregate do not belong to this one (run_stage2 sets them again)
  g->s2_ext = 0;
  if (!ext) { g->s2_m2.reset(); g->s2_prod.reset(); }
  // ... nor do its distinct pairs (run_count_distinct keeps this one's)
  g->cd_have = false;
  g->cd_n = 0;
  g->cd_id.reset(); g->cd_bits.reset();
  g->dp_parts_n = 0;
  PA_TRY(aggregate_impl(g, &val, agg_mask, deferred));
  if (g->pending) return PA_OK;
  if (had && prev_G != g->G) return set_err(PA_ERR_STATE, "group count changed between passes (%u vs %u)", prev_G, g->G);
  if (ext) PA_TRY(run_stage2(g, &val, ext));
  if (want_distinct) PA_TRY(run_count_distinct(g, &val));
  if (val.is_bool) {
    // the helper min / max columns are bytes, not Arrow booleans: only what was asked for stays fetchable
    keep_outputs(g, requested);
    if (extb) PA_TRY(run_bool_emit(g, extb));
  }
  // `val` may own device copies of host data: make sure the kernels reading them are done
  if (val.own_data.p) CUDA_TRY(cudaStreamSynchronize(g->stream));
  return PA_OK;
}

int pa_groupby_aggregate(pa_groupby* g, const struct ArrowDeviceArray* values, const struct ArrowSchema* value_schema,
                         uint32_t agg_mask) {
  return aggregate_entry(g, values, value_schema, agg_mask, false);
}

int pa_groupby_aggregate_async(pa_groupby* g, const struct ArrowDeviceArray* values, const struct ArrowSchema* value_schema,
                               uint32_t agg_mask) {
  return aggregate_entry(g, values, value_schema, agg_mask, true);
}

// NDFrame<T>::sum/mean/min/max/count/first/last/min_max/agg (/root/reference/src/ndframe.cpp:119-241): the whole
// column as ONE group (constant key generated on the device), through the same fused pass.
int pa_column_aggregate(const struct ArrowDeviceArray* values, const struct ArrowSchema* value_schema, uint32_t agg_mask,
                        int32_t skip_nulls, const pa_options* opt, pa_groupby** out) {
  if (!values || !value_schema || !out) return set_err(PA_ERR_INVALID, "pa_column_aggregate: null argument");
  if (agg_mask == 0 || (agg_mask & ~(PA_AGG_ALL | PA_AGG_STAGE2))) return set_err(PA_ERR_INVALID, "bad aggregate mask 0x%x", agg_mask);
  HandlePtr g(new pa_groupby());
  PA_TRY(handle_init(g.get(), opt));
  cudaStream_t st = g->stream;
  const int64_t n = values->array.length;
  if (n >= 0xFFFFFFFEll) return set_err(PA_ERR_NOT_IMPLEMENTED, "more than 2^32-2 rows per call; shard by row range");
  g->keys.resize(1);
  Column& k = g->keys[0];
  k.format = "l"; k.width = 8; k.vc = VC_I; k.n = n;
  PA_TRY(k.own_data.alloc(static_cast<size_t>(std::max<int64_t>(n, 1)) * 8, st));
  CUDA_TRY(cudaMemsetAsync(k.own_data.p, 0, static_cast<size_t>(std::max<int64_t>(n, 1)) * 8, st));
  k.data = k.own_data.p;
  g->n = n;
  PA_TRY(setup_keys(g.get()));
  const uint32_t positional = agg_mask & (PA_AGG_FIRST | PA_AGG_LAST);
  const bool patch = skip_nulls && positional && values->array.null_count != 0 && values->array.buffers[0] != nullptr && n > 0;
  if (!patch) {
    PA_TRY(aggregate_entry(g.get(), values, value_schema, agg_mask, false));
  } else {
    // first / last skip nulls here (arrow's scalar kernels), unlike GroupBy::first/last which are positional
    Column val;
    PA_TRY(load_column(values, value_schema, st, g->device, &val));
    if (val.is_bool) return set_err(PA_ERR_INVALID, "boolean columns aggregate with count / all / any only");
    PA_TRY(aggregate_impl(g.get(), &val, (agg_mask & PA_AGG_ALL) | PA_AGG_FIRST | PA_AGG_LAST));
    DevBuf range;
    PA_TRY(range.alloc(8, st));
    const uint32_t init[2] = {kNoRow, 0u};
    CUDA_TRY(cudaMemcpyAsync(range.p, init, 8, cudaMemcpyHostToDevice, st));
    const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, static_cast<int64_t>(g->num_sms) * 8)));
    k_valid_row_range<<<grid, 256, 0, st>>>(val.valid, val.bit_off, n, range.as<uint32_t>());
    CUDA_TRY(cudaGetLastError());
    if (g->G > 0) {
      k_apply_row_range<<<1, 1, 0, st>>>(range.as<uint32_t>(), g->res.first_row, g->res.last_row);
      CUDA_TRY(cudaGetLastError());
    }
    PA_TRY(run_emit(g.get(), &val, (agg_mask & PA_AGG_ALL) | PA_AGG_FIRST | PA_AGG_LAST));
    if (agg_mask & PA_AGG_STAGE2) PA_TRY(run_stage2(g.get(), &val, agg_mask & PA_AGG_STAGE2));
    CUDA_TRY(cudaStreamSynchronize(st));   // `val` / `range` may own device copies
  }
  *out = g.release();
  return PA_OK;
}

int pa_groupby_fetch(pa_groupby* g, uint32_t agg_bit, struct ArrowArray* out, struct ArrowSchema* out_schema) {
  if (!g || !out || !out_schema) return set_err(PA_ERR_INVALID, "null argument");
  PA_TRY(ensure_device(g));
  PA_TRY(finish_pending(g));
  for (auto& o : g->outs) {
    if (o.bit == agg_bit)
      return export_host(g->stream, o.format, o.width, g->G, o.values.p, o.nullable ? o.valid.as<uint32_t>() : nullptr, out, out_schema);
  }
  return set_err(PA_ERR_STATE, "aggregate 0x%x was not part of the last pa_groupby_aggregate call", agg_bit);
}

int pa_groupby_row_ids(pa_groupby* g, struct ArrowArray* out, struct ArrowSchema* out_schema) {
  if (!g || !out || !out_schema) return set_err(PA_ERR_INVALID, "null argument");
  if (g->merged) return set_err(PA_ERR_STATE, "row ids exist on the rank that holds the rows, not on a merged handle");
  PA_TRY(ensure_groups(g));
  PA_TRY(ensure_device(g));
  cudaStream_t st = g->stream;
  RowLookup lk;
  PA_TRY(build_row_lookup(g, &lk));
  DevBuf ids;
  PA_TRY(ids.alloc(static_cast<size_t>(std::max<int64_t>(g->n, 1)) * 4, st));
  lk.a.out = ids.as<uint32_t>();
  if (g->n) {
    const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((g->n + 255) / 256, static_cast<int64_t>(g->num_sms) * 16)));
    k_rowid_scan<<<grid, 256, 0, st>>>(lk.a);
    CUDA_TRY(cudaGetLastError());
  }
  return export_host(st, "I", 4, static_cast<uint32_t>(g->n), ids.p, nullptr, out, out_schema);
}

namespace {
// device-wide exclusive scan of a uint32 array in place (order.cuh)
int scan_u32(pa_groupby* g, uint32_t* data, uint64_t n, DevBuf* tile_sums) { return scan_u32_on(g, data, n, tile_sums); }

// ids -> stable counting sort by id (csort.cuh) -> (order, dest, offsets), cached on the handle
int ensure_groupings(pa_groupby* g) {
  if (g->have_groupings) return PA_OK;
  if (g->merged) return set_err(PA_ERR_STATE, "groupings exist on the rank that holds the rows, not on a merged handle");
  if (g->n >= (1ll << 31)) return set_err(PA_ERR_INVALID, "groupings use int32 offsets like the reference's ListArray<int32>: at most 2^31 - 1 rows");
  cudaStream_t st = g->stream;
  const uint32_t G = g->G;
  const int64_t n = g->n;
  CUDA_TRY(cudaEventRecord(g->ev[6], st));
  RowLookup lk;
  PA_TRY(build_row_lookup(g, &lk));
  DevBuf ids, keys_a, keys_b, pay_a, pay_b, counts, tile_sums;
  const size_t nb4 = static_cast<size_t>(std::max<int64_t>(n, 1)) * 4;
  PA_TRY(ids.alloc(nb4, st));
  PA_TRY(g->grp_order.alloc(nb4, st));
  PA_TRY(g->grp_dest.alloc(nb4, st));
  PA_TRY(g->grp_offsets.alloc((static_cast<size_t>(G) + 1) * 4, st));
  if (n > 0) {
    const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, static_cast<int64_t>(g->num_sms) * 16)));
    lk.a.out = ids.as<uint32_t>();
    k_rowid_scan<<<grid, 256, 0, st>>>(lk.a);
    CUDA_TRY(cudaGetLastError());
    int bits = 1;
    while (bits < 32 && (1ull << bits) < static_cast<uint64_t>(G)) ++bits;
    const int passes = (bits + CS_BITS - 1) / CS_BITS;
    const int64_t ntiles = (n + CS_TILE - 1) / CS_TILE;
    const int nb = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(ntiles, static_cast<int64_t>(g->num_sms) * 4)));
    const int64_t chunk = ((ntiles + nb - 1) / nb) * CS_TILE;
    PA_TRY(counts.alloc(sizeof(uint32_t) * CS_R * static_cast<size_t>(nb), st));
    if (passes > 1) {   // ping-pong buffers; the last pass writes its payload to grp_order and the sorted ids to keys_a / keys_b
      PA_TRY(keys_a.alloc(nb4, st));
      PA_TRY(pay_a.alloc(nb4, st));
      PA_TRY(keys_b.alloc(nb4, st));
      if (passes > 2) PA_TRY(pay_b.alloc(nb4, st));
    }
    static bool attr_set = false;
    if (!attr_set) {
      CUDA_TRY(cudaFuncSetAttribute(k_cs_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(CS_SMEM)));
      attr_set = true;
    }
    const uint32_t* in_keys = ids.as<uint32_t>();
    const uint32_t* in_pay = nullptr;
    for (int p = 0; p < passes; ++p) {
      const bool last = p == passes - 1;
      CsArgs a{};
      a.keys = in_keys; a.payload = in_pay; a.n = n; a.shift = p * CS_BITS; a.nb = nb; a.chunk = chunk;
      a.counts = counts.as<uint32_t>();
      DevBuf& ok = (p % 2 == 0) ? keys_a : keys_b;
      DevBuf& op = (p % 2 == 0) ? pay_a : pay_b;
      a.out_keys = last ? (passes > 1 ? ok.as<uint32_t>() : nullptr) : ok.as<uint32_t>();
      a.out_payload = last ? g->grp_order.as<uint32_t>() : op.as<uint32_t>();
      a.out_dest = last ? g->grp_dest.as<uint32_t>() : nullptr;
      k_cs_hist<<<nb, CS_THREADS, 0, st>>>(a);
      CUDA_TRY(cudaGetLastError());
      PA_TRY(scan_u32(g, counts.as<uint32_t>(), static_cast<uint64_t>(CS_R) * nb, &tile_sums));
      k_cs_scatter<<<nb, CS_THREADS, CS_SMEM, st>>>(a);
      CUDA_TRY(cudaGetLastError());
      if (last) {
        if (passes == 1) {
          k_cs_offsets<<<(G + 1 + 255) / 256, 256, 0, st>>>(counts.as<uint32_t>(), nb, G, n, g->grp_offsets.as<int32_t>());
        } else {
          k_group_offsets<<<grid, 256, 0, st>>>(a.out_keys, n, G, g->grp_offsets.as<int32_t>());
        }
        CUDA_TRY(cudaGetLastError());
      }
      in_keys = a.out_keys;
      in_pay = a.out_payload;
    }
  } else {
    CUDA_TRY(cudaMemsetAsync(g->grp_offsets.p, 0, (static_cast<size_t>(G) + 1) * 4, st));
  }
  CUDA_TRY(cudaEventRecord(g->ev[7], st));
  CUDA_TRY(cudaEventRecord(g->ev[8], st));
  CUDA_TRY(cudaEventRecord(g->ev[9], st));
  CUDA_TRY(cudaStreamSynchronize(st));   // the sort buffers above are released here
  g->have_groupings = true;
  return PA_OK;
}
}  // namespace

// unique() of a utf8 / large_utf8 key: the bytes of col's row rows[g] for every group g, in group order — a local
// handle's first rows in its key column, or a merged handle's compacted representatives — as utf8 (large: large_utf8)
// with int32 offsets (a result of more than 2 GiB of distinct strings is refused).  kind[g] == KK_NULL: group g's
// string is null (the key kinds, or a hashed composite key's column at the first rows).
static int unique_strings(pa_groupby* g, const StrCol& col, const uint32_t* rows, const uint8_t* kind, bool large, struct ArrowArray* out,
                          struct ArrowSchema* out_schema) {
  cudaStream_t st = g->stream;
  const uint32_t G = g->G;
  DevBuf offs, tile_sums, bytes, valid;
  PA_TRY(offs.alloc(static_cast<size_t>(G + 1) * 4, st));
  k_str_lengths<<<(G + 1 + 255) / 256, 256, 0, st>>>(col, rows, kind, G, offs.as<uint32_t>());
  CUDA_TRY(cudaGetLastError());
  uint64_t total64 = 0;
  {
    DevBuf tot;
    PA_TRY(tot.alloc(8, st));
    CUDA_TRY(cudaMemsetAsync(tot.p, 0, 8, st));
    if (G) k_sum_u32<<<std::min<uint32_t>((G + 255) / 256, 1024u), 256, 0, st>>>(offs.as<uint32_t>(), G, tot.as<unsigned long long>());
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(&total64, tot.p, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
  }
  if (total64 > 0x7FFFFFFFull) return set_err(PA_ERR_NOT_IMPLEMENTED, "distinct utf8 keys total %llu bytes; int32 offsets hold 2 GiB", (unsigned long long)total64);
  PA_TRY(scan_u32(g, offs.as<uint32_t>(), static_cast<uint64_t>(G) + 1, &tile_sums));
  PA_TRY(bytes.alloc(std::max<uint64_t>(total64, 1), st));
  PA_TRY(valid.alloc(((static_cast<size_t>(G) + 31) / 32 + 1) * 4, st));
  if (G) {
    k_str_gather<<<(static_cast<uint64_t>(G) * 32 + 255) / 256, 256, 0, st>>>(col, rows, kind, G, offs.as<uint32_t>(), bytes.as<uint8_t>());
    CUDA_TRY(cudaGetLastError());
    k_kind_validity<<<(G + 31) / 32 * 32 / 256 + 1, 256, 0, st>>>(kind, G, valid.as<uint32_t>());
    CUDA_TRY(cudaGetLastError());
  }
  auto* priv = new ExportPriv();
  const size_t words = (static_cast<size_t>(G) + 31) / 32;
  priv->bufs[0] = malloc(std::max<size_t>(words * 4, 64));
  priv->bufs[1] = malloc(std::max<size_t>((static_cast<size_t>(G) + 1) * 4, 64));
  priv->bufs[2] = malloc(std::max<size_t>(total64, 64));
  cudaError_t e = cudaMemcpyAsync(priv->bufs[1], offs.p, (static_cast<size_t>(G) + 1) * 4, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess && G) e = cudaMemcpyAsync(priv->bufs[0], valid.p, words * 4, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess && total64) e = cudaMemcpyAsync(priv->bufs[2], bytes.p, total64, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) {
    free(priv->bufs[0]); free(priv->bufs[1]); free(priv->bufs[2]); delete priv;
    return set_err(PA_ERR_CUDA, "result copy failed: %s", cudaGetErrorString(e));
  }
  int64_t set = 0;
  for (size_t i = 0; i < words; ++i) set += __builtin_popcount(static_cast<const uint32_t*>(priv->bufs[0])[i]);
  const int64_t null_count = static_cast<int64_t>(G) - set;
  if (null_count == 0) { free(priv->bufs[0]); priv->bufs[0] = nullptr; }
  if (large) {   // large_utf8 in, large_utf8 out (int64 offsets, widened on the host: G + 1 numbers)
    int64_t* wide = static_cast<int64_t*>(malloc(std::max<size_t>((static_cast<size_t>(G) + 1) * 8, 64)));
    for (size_t i = 0; i <= G; ++i) wide[i] = static_cast<const uint32_t*>(priv->bufs[1])[i];
    free(priv->bufs[1]);
    priv->bufs[1] = wide;
  }
  for (int i = 0; i < 3; ++i) priv->ptrs[i] = priv->bufs[i];
  memset(out, 0, sizeof *out);
  out->length = G;
  out->null_count = null_count;
  out->n_buffers = 3;
  out->buffers = priv->ptrs;
  out->release = release_array;
  out->private_data = priv;
  memset(out_schema, 0, sizeof *out_schema);
  auto* f = new std::string(large ? "U" : "u");
  out_schema->format = f->c_str();
  out_schema->name = "";
  out_schema->flags = ARROW_FLAG_NULLABLE;
  out_schema->release = release_schema;
  out_schema->private_data = f;
  return PA_OK;
}

int pa_groupby_groupings(pa_groupby* g, struct ArrowArray* offsets, struct ArrowSchema* offsets_schema,
                         struct ArrowArray* rows, struct ArrowSchema* rows_schema) {
  if (!g || !offsets || !offsets_schema) return set_err(PA_ERR_INVALID, "null argument");
  if ((rows == nullptr) != (rows_schema == nullptr)) return set_err(PA_ERR_INVALID, "rows and rows_schema go together");
  PA_TRY(ensure_groups(g));
  PA_TRY(ensure_device(g));
  PA_TRY(ensure_groupings(g));
  PA_TRY(export_host(g->stream, "i", 4, g->G + 1, g->grp_offsets.p, nullptr, offsets, offsets_schema));
  if (rows) PA_TRY(export_host(g->stream, "i", 4, static_cast<uint32_t>(g->n), g->grp_order.p, nullptr, rows, rows_schema));
  return PA_OK;
}

int pa_groupby_take_grouped(pa_groupby* g, const struct ArrowDeviceArray* column, const struct ArrowSchema* schema,
                            struct ArrowArray* out, struct ArrowSchema* out_schema) {
  if (!g || !column || !schema || !out || !out_schema) return set_err(PA_ERR_INVALID, "null argument");
  PA_TRY(ensure_groups(g));
  PA_TRY(ensure_device(g));
  PA_TRY(ensure_groupings(g));
  cudaStream_t st = g->stream;
  Column col;
  PA_TRY(load_column(column, schema, st, g->device, &col));
  if (col.n != g->n) return set_err(PA_ERR_INVALID, "column has %lld rows, keys have %lld", (long long)col.n, (long long)g->n);
  if (schema->dictionary) return set_err(PA_ERR_INVALID, "dictionary-encoded columns: gather the indices, keep the dictionary");
  const int64_t n = g->n;
  const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, static_cast<int64_t>(g->num_sms) * 16)));
  const size_t words = (static_cast<size_t>(n) + 31) / 32 + 1;
  DevBuf vals, valid;
  if (col.is_bool) {
    // bit-packed values: gathered bit by bit from the packed input (load_column keeps it in own_bits for host
    // inputs; device inputs are read in place)
    const ArrowArray& arr = column->array;
    const uint8_t* bits = col.own_bits.p ? col.own_bits.as<uint8_t>() : static_cast<const uint8_t*>(arr.buffers[1]);
    const int64_t boff = col.own_bits.p ? arr.offset % 8 : arr.offset;
    PA_TRY(vals.alloc(words * 4, st));
    if (col.valid) PA_TRY(valid.alloc(words * 4, st));
    if (n > 0) {
      CUDA_TRY(cudaEventRecord(g->ev[8], st));
      k_take_bits<<<grid, 256, 0, st>>>(bits, boff, g->grp_order.as<uint32_t>(), n, vals.as<uint32_t>());
      CUDA_TRY(cudaGetLastError());
      if (col.valid) {
        k_take_bits<<<grid, 256, 0, st>>>(col.valid, col.bit_off, g->grp_order.as<uint32_t>(), n, valid.as<uint32_t>());
        CUDA_TRY(cudaGetLastError());
      }
      CUDA_TRY(cudaEventRecord(g->ev[9], st));
    }
    return export_host(st, "b", 1, static_cast<uint32_t>(n), vals.p, col.valid ? valid.as<uint32_t>() : nullptr, out, out_schema);
  }
  PA_TRY(vals.alloc(static_cast<size_t>(std::max<int64_t>(n, 1)) * col.width, st));
  if (col.valid) {
    PA_TRY(valid.alloc(words * 4, st));
    CUDA_TRY(cudaMemsetAsync(valid.p, 0, words * 4, st));
  }
  if (n > 0) {
    TakeScatterArgs a{};
    a.col = col.data;
    a.valid = col.valid;
    a.bit_off = col.bit_off;
    a.width = col.width;
    a.dest = g->grp_dest.as<uint32_t>();
    a.n = n;
    a.out = vals.p;
    a.out_valid = col.valid ? valid.as<uint32_t>() : nullptr;
    CUDA_TRY(cudaEventRecord(g->ev[8], st));
    k_take_scatter<<<grid, 256, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(g->ev[9], st));
  }
  return export_host(st, col.format, col.width, static_cast<uint32_t>(n), vals.p, col.valid ? valid.as<uint32_t>() : nullptr, out, out_schema);
}

int pa_groupby_groupings_timing(pa_groupby* g, double* build_ms, double* take_ms) {
  if (!g) return set_err(PA_ERR_INVALID, "null argument");
  if (!g->have_groupings) return set_err(PA_ERR_STATE, "no groupings were built on this handle");
  PA_TRY(ensure_device(g));
  CUDA_TRY(cudaEventSynchronize(g->ev[9]));
  float t = 0;
  if (build_ms) { CUDA_TRY(cudaEventElapsedTime(&t, g->ev[6], g->ev[7])); *build_ms = t; }
  if (take_ms) { CUDA_TRY(cudaEventElapsedTime(&t, g->ev[8], g->ev[9])); *take_ms = t; }
  return PA_OK;
}

int pa_groupby_first_rows(pa_groupby* g, struct ArrowArray* out, struct ArrowSchema* out_schema) {
  if (!g || !out || !out_schema) return set_err(PA_ERR_INVALID, "null argument");
  PA_TRY(ensure_groups(g));
  PA_TRY(ensure_device(g));
  if (g->merged) return export_host(g->stream, "L", 8, g->G, g->m_first_row_g.p, nullptr, out, out_schema);
  PA_TRY(export_host(g->stream, "I", 4, g->G, g->res.first_row, nullptr, out, out_schema));
  // widen to uint64 and add the shard's row base on the host (G values)
  auto* priv = static_cast<ExportPriv*>(out->private_data);
  const uint32_t* src = static_cast<const uint32_t*>(priv->bufs[1]);
  uint64_t* wide = static_cast<uint64_t*>(malloc(std::max<size_t>(static_cast<size_t>(g->G) * 8, 64)));
  for (uint32_t i = 0; i < g->G; ++i) wide[i] = static_cast<uint64_t>(g->opt.row_base) + src[i];
  free(priv->bufs[1]);
  priv->bufs[1] = wide;
  priv->ptrs[1] = wide;
  delete static_cast<std::string*>(out_schema->private_data);
  auto* f = new std::string("L");
  out_schema->format = f->c_str();
  out_schema->private_data = f;
  return PA_OK;
}

int pa_groupby_last_timing(pa_groupby* g, double* total_ms, double stage_ms[4]) {
  if (!g) return set_err(PA_ERR_INVALID, "null argument");
  PA_TRY(ensure_device(g));
  PA_TRY(finish_pending(g));
  CUDA_TRY(cudaEventSynchronize(g->ev[4]));
  float t = 0;
  CUDA_TRY(cudaEventElapsedTime(&t, g->ev[0], g->ev[4]));
  if (total_ms) *total_ms = t;
  if (stage_ms) {
    float a = 0, b = 0, c = 0, d = 0;
    CUDA_TRY(cudaEventElapsedTime(&a, g->ev[0], g->ev[1]));
    CUDA_TRY(cudaEventElapsedTime(&b, g->ev[1], g->ev[2]));
    CUDA_TRY(cudaEventElapsedTime(&c, g->ev[2], g->ev[3]));
    CUDA_TRY(cudaEventElapsedTime(&d, g->ev[3], g->ev[4]));
    stage_ms[0] = a; stage_ms[1] = b; stage_ms[2] = c; stage_ms[3] = d;
  }
  return PA_OK;
}

int pa_groupby_last_path(pa_groupby* g, int32_t* path, int32_t* kernel_launches) {
  if (!g) return set_err(PA_ERR_INVALID, "null argument");
  PA_TRY(finish_pending(g));
  if (path) *path = g->last_path;
  if (kernel_launches) *kernel_launches = g->last_launches;
  return PA_OK;
}

int pa_groupby_last_detail(pa_groupby* g, int32_t detail[4]) {
  if (!g || !detail) return set_err(PA_ERR_INVALID, "null argument");
  PA_TRY(finish_pending(g));
  detail[0] = g->last_mode; detail[1] = g->last_rlog; detail[2] = g->last_passes; detail[3] = 0;
  return PA_OK;
}

int pa_groupby_sync(pa_groupby* g) {
  if (!g) return set_err(PA_ERR_INVALID, "null argument");
  PA_TRY(ensure_device(g));
  PA_TRY(finish_pending(g));
  CUDA_TRY(cudaStreamSynchronize(g->stream));
  return PA_OK;
}

void pa_groupby_destroy(pa_groupby* g) {
  if (!g) return;
  if (g->merged && !g->own_stream && g->poolable) {
    // recycle: nothing is freed, so no synchronisation is needed either (stream order protects the buffers)
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    if (g_merge_pool.size() < 4) {
      g->outs.clear();
      g->have_groups = false;
      g->pending_merge = false;
      g->G = 0;
      g_merge_pool.push_back(g);
      return;
    }
  }
  cudaSetDevice(g->device);
  cudaStreamSynchronize(g->stream);
  g->outs.clear();
  cudaStream_t st = g->stream;
  const bool own = g->own_stream;
  for (auto& e : g->ev) if (e) cudaEventDestroy(e);
  delete g;   // DevBufs free on `st`
  if (own) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
}

int pa_resample_create(const struct ArrowDeviceArray* index, const struct ArrowSchema* index_schema, int64_t freq_ns,
                       int32_t closed_right, int32_t label_right, int32_t origin, int64_t origin_custom_ns,
                       int64_t offset_ns, const pa_options* opt, pa_groupby** out) {
  if (!index || !index_schema || !out) return set_err(PA_ERR_INVALID, "pa_resample_create: null argument");
  if (freq_ns <= 0) return set_err(PA_ERR_INVALID, "FREQ must be positive");   // core.cpp:319-322
  HandlePtr g(new pa_groupby());
  PA_TRY(handle_init(g.get(), opt));
  g->keys.resize(1);
  Column& ix = g->keys[0];
  PA_TRY(load_column(index, index_schema, g->stream, g->device, &ix));
  const char* f = index_schema->format;
  const bool is_ts = f && f[0] == 't' && f[1] == 's';
  if (!(is_ts || (f && f[0] == 'l')) || ix.width != 8)
    return set_err(PA_ERR_INVALID, "axis must be a TimestampArray but got array of type '%s'", f ? f : "?");  // resample.cpp:213-216
  if (ix.valid) return set_err(PA_ERR_NOT_IMPLEMENTED, "resample: null timestamps are not supported");
  int64_t ticks_per_day = 86400LL * 1000000000LL;
  int64_t ns_per_tick = 1;
  if (is_ts) {
    switch (f[2]) {
      case 's': ticks_per_day = 86400LL; ns_per_tick = 1000000000LL; break;
      case 'm': ticks_per_day = 86400LL * 1000; ns_per_tick = 1000000LL; break;
      case 'u': ticks_per_day = 86400LL * 1000000; ns_per_tick = 1000LL; break;
      default: break;
    }
  }
  // freq / offset / custom origin arrive in nanoseconds; the bucket arithmetic runs in index ticks
  if (ns_per_tick != 1) {
    if (freq_ns % ns_per_tick || offset_ns % ns_per_tick || (origin == 5 && origin_custom_ns % ns_per_tick))
      return set_err(PA_ERR_INVALID, "resample: freq / offset / origin are not whole multiples of the index unit ('%s')", f);
    freq_ns /= ns_per_tick;
    offset_ns /= ns_per_tick;
    origin_custom_ns /= ns_per_tick;
  }
  g->n = ix.n;
  if (g->n >= 0xFFFFFFFELL) return set_err(PA_ERR_NOT_IMPLEMENTED, "more than 2^32-2 rows per call; shard by row range");
  g->resample = true;
  g->index_format = f;
  g->fields.assign(1, KeyField{});
  g->key_data = ix.data;
  g->key_width = 8;
  g->rs = ResampleSpec{};
  g->rs.freq = freq_ns;
  g->rs.closed_right = closed_right != 0;
  g->rs.label_off = label_right ? freq_ns : 0;
  if (g->n > 0) {
    int64_t ends[2];
    CUDA_TRY(cudaMemcpyAsync(&ends[0], ix.data, 8, cudaMemcpyDeviceToHost, g->stream));
    CUDA_TRY(cudaMemcpyAsync(&ends[1], static_cast<const int64_t*>(ix.data) + (g->n - 1), 8, cudaMemcpyDeviceToHost, g->stream));
    CUDA_TRY(cudaStreamSynchronize(g->stream));
    if (ends[1] < ends[0]) return set_err(PA_ERR_INVALID, "resample: the index must be sorted ascending");
    int64_t first, last;
    anchor_range(ends[0], ends[1], freq_ns, closed_right != 0, origin, origin_custom_ns, offset_ns, ticks_per_day, &first, &last);
    if (first >= last) return set_err(PA_ERR_INVALID, "start date has to be less than end date");  // core.cpp:314-317
    g->rs.first = first;
    g->rs.nbins = (last - first) / freq_ns;
    if (g->n < g->rs.nbins) return set_err(PA_ERR_NOT_IMPLEMENTED, "upSampling is not implemented.");  // resample.h:102-105
  }
  *out = g.release();
  return PA_OK;
}

// pd::resample with a DateOffset rule (makeGroupInfo's DateOffset branch, /root/reference/src/resample.cpp:248-267;
// DateOffset::add, core.cpp:12-60; date_range + switchFunction, core.cpp:175-265; adjustBinEdges, resample.cpp:180-200).
// The host computes the O(#buckets) binner / edge / label arrays; the rows are reduced by the same sorted-run kernel
// as the fixed-width rules, which looks a bucket up in the edge array only where a new run of rows begins.
namespace {
int64_t days_from_civil(int64_t y, int m, int d) {       // proleptic Gregorian, days since 1970-01-01
  y -= m <= 2;
  const int64_t era = (y >= 0 ? y : y - 399) / 400;
  const int64_t yoe = y - era * 400;
  const int64_t doy = (153 * (m + (m > 2 ? -3 : 9)) + 2) / 5 + d - 1;
  const int64_t doe = yoe * 365 + yoe / 4 - yoe / 100 + doy;
  return era * 146097 + doe - 719468;
}
void civil_from_days(int64_t z, int64_t* y, int* m, int* d) {
  z += 719468;
  const int64_t era = (z >= 0 ? z : z - 146096) / 146097;
  const int64_t doe = z - era * 146097;
  const int64_t yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
  const int64_t doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
  const int64_t mp = (5 * doy + 2) / 153;
  *d = static_cast<int>(doy - (153 * mp + 2) / 5 + 1);
  *m = static_cast<int>(mp < 10 ? mp + 3 : mp - 9);
  *y = yoe + era * 400 + (*m <= 2);
}
// DateOffset::add for the rule types date_range accepts; the day of the month only survives for Day / WeekStart,
// the others snap to the first day of a month, so boost's end-of-month rules never come into play.
int64_t offset_add(int64_t day, int type, int64_t k) {
  if (type == PA_OFFSET_DAY) return day + k;
  if (type == PA_OFFSET_WEEK_START) return day + 7 * k;
  int64_t y; int m, d;
  civil_from_days(day, &y, &m, &d);
  int64_t ym = y * 12 + (m - 1);
  if (type == PA_OFFSET_MONTH_START) ym += k;
  else if (type == PA_OFFSET_QUARTER_START) { ym += 3 * k; ym = floor_div(ym, 3) * 3; }
  else /* YEAR_START */ { ym += 12 * k; ym = floor_div(ym, 12) * 12; }
  return days_from_civil(floor_div(ym, 12), static_cast<int>(ym - floor_div(ym, 12) * 12) + 1, 1);
}
}  // namespace

int pa_resample_create_calendar(const struct ArrowDeviceArray* index, const struct ArrowSchema* index_schema, int32_t offset_type,
                                int32_t multiplier, int32_t closed_right, int32_t label_right, const pa_options* opt,
                                pa_groupby** out) {
  if (!index || !index_schema || !out) return set_err(PA_ERR_INVALID, "pa_resample_create_calendar: null argument");
  if (multiplier < 1) return set_err(PA_ERR_INVALID, "FREQ must be >= 1");                                   // core.cpp:186-189
  switch (offset_type) {
    case PA_OFFSET_DAY: case PA_OFFSET_WEEK_START: case PA_OFFSET_MONTH_START: case PA_OFFSET_QUARTER_START: case PA_OFFSET_YEAR_START: break;
    case PA_OFFSET_MONTH_END: return set_err(PA_ERR_NOT_IMPLEMENTED, "MonthEnd not supported use arrow month().groupby()");       // core.cpp:243-260
    case PA_OFFSET_QUARTER_END: return set_err(PA_ERR_NOT_IMPLEMENTED, "QuarterEnd not supported use arrow quarter().groupby()");
    case PA_OFFSET_WEEK_END: return set_err(PA_ERR_NOT_IMPLEMENTED, "WeekEnd not supported use arrow weeks().groupby()");
    case PA_OFFSET_YEAR_END: return set_err(PA_ERR_NOT_IMPLEMENTED, "YearEnd not supported use arrow year().groupby()");
    default: return set_err(PA_ERR_INVALID, "unknown DateOffset type %d", offset_type);
  }
  if (!closed_right) return set_err(PA_ERR_NOT_IMPLEMENTED, "closed_left is not currently supported by DateOffset");   // resample.cpp:256-258
  HandlePtr g(new pa_groupby());
  PA_TRY(handle_init(g.get(), opt));
  g->keys.resize(1);
  Column& ix = g->keys[0];
  PA_TRY(load_column(index, index_schema, g->stream, g->device, &ix));
  const char* f = index_schema->format;
  if (!(f && f[0] == 't' && f[1] == 's') || ix.width != 8)
    return set_err(PA_ERR_INVALID, "axis must be a TimestampArray but got array of type '%s'", f ? f : "?");   // resample.cpp:213-216
  if (f[2] != 'n') return set_err(PA_ERR_NOT_IMPLEMENTED, "resample by a DateOffset rule needs a timestamp[ns] index (the reference's bins and labels are nanoseconds)");
  if (ix.valid) return set_err(PA_ERR_NOT_IMPLEMENTED, "resample: null timestamps are not supported");
  g->n = ix.n;
  if (g->n >= 0xFFFFFFFELL) return set_err(PA_ERR_NOT_IMPLEMENTED, "more than 2^32-2 rows per call; shard by row range");
  g->resample = true;
  g->index_format = f;
  g->fields.assign(1, KeyField{});
  g->key_data = ix.data;
  g->key_width = 8;
  g->rs = ResampleSpec{};
  g->rs.closed_right = 1;
  if (g->n > 0) {
    constexpr int64_t kDay = 86400LL * 1000000000LL;
    int64_t ends[2];
    CUDA_TRY(cudaMemcpyAsync(&ends[0], ix.data, 8, cudaMemcpyDeviceToHost, g->stream));
    CUDA_TRY(cudaMemcpyAsync(&ends[1], static_cast<const int64_t*>(ix.data) + (g->n - 1), 8, cudaMemcpyDeviceToHost, g->stream));
    CUDA_TRY(cudaStreamSynchronize(g->stream));
    if (ends[1] < ends[0]) return set_err(PA_ERR_INVALID, "resample: the index must be sorted ascending");
    const int64_t first_day = floor_div(ends[0], kDay), last_day = floor_div(ends[1], kDay);
    const int64_t start = offset_add(first_day, offset_type, -static_cast<int64_t>(multiplier));
    const int64_t stop = offset_add(last_day, offset_type, multiplier);
    if (start >= stop) return set_err(PA_ERR_INVALID, "start date has to be less than end date");              // core.cpp:181-184
    if (offset_type == PA_OFFSET_QUARTER_START) {
      int64_t y; int m, d;
      civil_from_days(start, &y, &m, &d);
      if (m / 3 != 0) return set_err(PA_ERR_INVALID, "A quarter freq requires month is on a quarter, +/- with DateOffset");   // core.cpp:247-250
    }
    // date_range(first - freq, last + freq, freq): the iterator steps `multiplier` units from `start` while <= stop
    std::vector<int64_t> binner;
    for (int64_t i = 0;; ++i) {
      int64_t day;
      if (offset_type == PA_OFFSET_DAY) day = start + i * multiplier;
      else if (offset_type == PA_OFFSET_WEEK_START) day = start + 7 * i * multiplier;
      else day = offset_add(start, offset_type, i * multiplier);
      if (day > stop) break;
      binner.push_back(day * kDay);
      if (binner.size() > (1u << 28)) return set_err(PA_ERR_INVALID, "resample: too many buckets");
    }
    std::vector<int64_t> edges(binner);
    if (!(offset_type == PA_OFFSET_DAY && multiplier == 1)) {                                                 // adjustBinEdges
      for (auto& e : edges) e += kDay - 1;
      if (edges.size() >= 2 && edges[edges.size() - 2] > ends[1]) { edges.pop_back(); binner.pop_back(); }
    }
    if (edges.size() < 2) return set_err(PA_ERR_INVALID, "Invalid length for values or for binner");
    if (ends[0] < edges.front()) return set_err(PA_ERR_INVALID, "Values falls before first bin");             // resample.cpp:33-41
    if (ends[1] > edges.back()) return set_err(PA_ERR_INVALID, "Values falls after last bin");
    const int64_t nbins = static_cast<int64_t>(edges.size()) - 1;
    if (g->n < nbins) return set_err(PA_ERR_NOT_IMPLEMENTED, "upSampling is not implemented.");               // resample.h:102-105
    std::vector<int64_t> labels(static_cast<size_t>(nbins));
    for (int64_t i = 0; i < nbins; ++i) labels[i] = binner[static_cast<size_t>(i) + (label_right ? 1 : 0)];
    // bin i = (edges[i], edges[i+1]] on ts = [edges[i], edges[i+1]) on ts' = ts - 1; a value equal to edges[0] passes
    // the reference's range check and lands in bin 0
    edges[0] -= 1;
    PA_TRY(g->rs_edges.alloc(edges.size() * 8, g->stream));
    PA_TRY(g->rs_labels.alloc(labels.size() * 8, g->stream));
    CUDA_TRY(cudaMemcpyAsync(g->rs_edges.p, edges.data(), edges.size() * 8, cudaMemcpyHostToDevice, g->stream));
    CUDA_TRY(cudaMemcpyAsync(g->rs_labels.p, labels.data(), labels.size() * 8, cudaMemcpyHostToDevice, g->stream));
    CUDA_TRY(cudaStreamSynchronize(g->stream));
    g->rs.first = edges[0];
    g->rs.freq = kDay;
    g->rs.nbins = nbins;
    g->rs.edges = g->rs_edges.as<int64_t>();
    g->rs.labels = g->rs_labels.as<int64_t>();
  }
  *out = g.release();
  return PA_OK;
}

// DataFrame::downsample (/root/reference/src/dataframe.cpp:1265-1290): per-row label = Floor/CeilTemporal(index)
// computed on the device (temporal.cuh), then the ordinary hash group-by on the labels.
int pa_downsample_create(const struct ArrowDeviceArray* index, const struct ArrowSchema* index_schema, int32_t multiple,
                         char unit, int32_t closed_label_right, int32_t week_starts_monday, int32_t calendar_based_origin,
                         const pa_options* opt, pa_groupby** out) {
  if (!index || !index_schema || !out) return set_err(PA_ERR_INVALID, "pa_downsample_create: null argument");
  if (multiple < 1) return set_err(PA_ERR_INVALID, "Invalid time offset: multiple must be >= 1");
  const char* units = "NULSTHDWMQY";
  if (!unit || !strchr(units, unit)) return set_err(PA_ERR_INVALID, "Invalid time offset unit '%c'", unit ? unit : '?');
  const char* f = index_schema->format;
  if (!f || f[0] != 't' || f[1] != 's') return set_err(PA_ERR_INVALID, "axis must be a TimestampArray but got array of type '%s'", f ? f : "?");
  HandlePtr g(new pa_groupby());
  PA_TRY(handle_init(g.get(), opt));
  cudaStream_t st = g->stream;
  Column ix;
  PA_TRY(load_column(index, index_schema, st, g->device, &ix));
  int64_t tps = 1000000000LL;
  switch (f[2]) {
    case 's': tps = 1; break;
    case 'm': tps = 1000; break;
    case 'u': tps = 1000000; break;
    default: break;
  }
  const bool calendar = unit == 'W' || unit == 'M' || unit == 'Q' || unit == 'Y';
  // the reference's W / M / Q / Y branch subtracts one day and re-types the labels as timestamp[ns]
  // (dataframe.cpp:1279-1287); other resolutions would change meaning there
  if (calendar && tps != 1000000000LL) return set_err(PA_ERR_NOT_IMPLEMENTED, "downsample by W / M / Q / Y needs a timestamp[ns] index");
  TemporalSpec spec{};
  spec.multiple = multiple;
  spec.unit = unit;
  spec.ceil = closed_label_right ? 1 : 0;
  spec.week_starts_monday = week_starts_monday ? 1 : 0;
  spec.calendar_origin = calendar_based_origin ? 1 : 0;
  spec.ticks_per_sec = tps;
  spec.post_shift = calendar ? -86400LL * tps : 0;
  g->keys.resize(1);
  Column& k = g->keys[0];
  k.format = calendar ? "tsn:" : f;
  k.width = 8; k.vc = VC_I; k.n = ix.n;
  PA_TRY(k.own_data.alloc(static_cast<size_t>(std::max<int64_t>(ix.n, 1)) * 8, st));
  if (ix.n > 0) {
    const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((ix.n + 255) / 256, static_cast<int64_t>(g->num_sms) * 16)));
    k_temporal_labels<<<grid, 256, 0, st>>>(static_cast<const int64_t*>(ix.data), ix.valid, ix.bit_off, ix.n, spec, k.own_data.as<int64_t>());
    CUDA_TRY(cudaGetLastError());
  }
  k.data = k.own_data.p;
  if (ix.valid) {   // null timestamps stay null labels: their own group, like any null key
    if (ix.own_valid.p) k.own_valid = std::move(ix.own_valid);
    k.valid = ix.valid;
    k.bit_off = ix.bit_off;
  }
  g->n = ix.n;
  if (g->n >= 0xFFFFFFFEll) return set_err(PA_ERR_NOT_IMPLEMENTED, "more than 2^32-2 rows per call; shard by row range");
  PA_TRY(setup_keys(g.get()));
  CUDA_TRY(cudaStreamSynchronize(st));   // `ix` may own the device copy of a host index
  *out = g.release();
  return PA_OK;
}

// ---- ingest: one host Arrow array -> device-resident ArrowDeviceArray (SURVEY §8f rank 4) ----
// What DataFrame::readBinary / readParquet (dataframe.cpp:757-791, 646-683) produce are host Arrow arrays inside an IPC
// blob or a decoded table; this puts a column on the device ONCE (pageable memory through the pinned staging pipeline of
// h2d_copy) and hands back an ArrowDeviceArray(CUDA) that every other entry point uses in place, so that the
// constructor and every aggregate after it stop paying PCIe.
namespace {
struct DevArrayPriv {
  void* owned[3] = {nullptr, nullptr, nullptr};
  const void* bufs[3] = {nullptr, nullptr, nullptr};
};
void dev_array_release(struct ArrowArray* a) {
  if (!a || !a->release) return;
  auto* p = static_cast<DevArrayPriv*>(a->private_data);
  if (p) {
    for (void* q : p->owned) if (q) cudaFree(q);
    delete p;
  }
  a->release = nullptr;
}
}  // namespace

int pa_column_to_device(const struct ArrowDeviceArray* host, const struct ArrowSchema* schema, const pa_options* opt,
                        struct ArrowDeviceArray* out) {
  if (!host || !schema || !out || !schema->format) return set_err(PA_ERR_INVALID, "pa_column_to_device: null argument");
  if (host->device_type != ARROW_DEVICE_CPU && host->device_type != ARROW_DEVICE_CUDA_HOST)
    return set_err(PA_ERR_INVALID, "pa_column_to_device: the input must be a host array");
  if (schema->dictionary) return set_err(PA_ERR_NOT_IMPLEMENTED, "pa_column_to_device: dictionary-encoded columns (ingest the indices)");
  const ArrowArray& a = host->array;
  const char f0 = schema->format[0];
  const bool is_str = f0 == 'u' || f0 == 'U';
  const bool is_bool = f0 == 'b';
  int width = 0, vc = 0;
  if (!is_str) PA_TRY(parse_format(schema->format, &width, &vc));
  if (a.n_buffers < (is_str ? 3 : 2)) return set_err(PA_ERR_INVALID, "unexpected buffer count %lld for format '%s'", (long long)a.n_buffers, schema->format);
  int device = 0;
  if (opt && opt->device >= 0) device = opt->device; else CUDA_TRY(cudaGetDevice(&device));
  CUDA_TRY(cudaSetDevice(device));
  cudaStream_t st = opt && opt->cuda_stream ? static_cast<cudaStream_t>(opt->cuda_stream) : nullptr;
  std::unique_ptr<DevArrayPriv> p(new DevArrayPriv());
  struct Guard { DevArrayPriv* p; ~Guard() { if (p) for (void* q : p->owned) if (q) cudaFree(q); } } guard{p.get()};
  const int64_t k = a.offset % 8, start = a.offset - k, n = a.length;
  const bool has_nulls = a.null_count != 0 && a.buffers[0] != nullptr;
  const size_t bit_bytes = static_cast<size_t>((k + n + 7) / 8);
  if (has_nulls) {
    CUDA_TRY(cudaMalloc(&p->owned[0], std::max<size_t>(bit_bytes, 16)));
    PA_TRY(h2d_copy(p->owned[0], static_cast<const uint8_t*>(a.buffers[0]) + start / 8, bit_bytes, st));
    p->bufs[0] = p->owned[0];
  }
  if (is_str) {
    const int ow = f0 == 'U' ? 8 : 4;
    const char* offs = static_cast<const char*>(a.buffers[1]) + start * ow;
    const size_t obytes = static_cast<size_t>(k + n + 1) * ow;
    CUDA_TRY(cudaMalloc(&p->owned[1], std::max<size_t>(obytes, 16)));
    int64_t first = 0, last = 0;
    if (a.buffers[1]) {
      PA_TRY(h2d_copy(p->owned[1], offs, obytes, st));
      first = ow == 8 ? reinterpret_cast<const int64_t*>(offs)[0] : reinterpret_cast<const int32_t*>(offs)[0];
      last = ow == 8 ? reinterpret_cast<const int64_t*>(offs)[k + n] : reinterpret_cast<const int32_t*>(offs)[k + n];
    } else {
      CUDA_TRY(cudaMemsetAsync(p->owned[1], 0, obytes, st));
    }
    CUDA_TRY(cudaMalloc(&p->owned[2], static_cast<size_t>(std::max<int64_t>(last - first, 16))));
    if (last > first) PA_TRY(h2d_copy(p->owned[2], static_cast<const uint8_t*>(a.buffers[2]) + first, static_cast<size_t>(last - first), st));
    p->bufs[1] = p->owned[1];
    p->bufs[2] = static_cast<const uint8_t*>(p->owned[2]) - first;     // offsets stay absolute
  } else if (is_bool) {
    CUDA_TRY(cudaMalloc(&p->owned[1], std::max<size_t>(bit_bytes, 16)));
    if (a.buffers[1]) PA_TRY(h2d_copy(p->owned[1], static_cast<const uint8_t*>(a.buffers[1]) + start / 8, bit_bytes, st));
    p->bufs[1] = p->owned[1];
  } else {
    const size_t bytes = static_cast<size_t>(k + n) * width;
    CUDA_TRY(cudaMalloc(&p->owned[1], std::max<size_t>(bytes, 16)));
    if (a.buffers[1]) PA_TRY(h2d_copy(p->owned[1], static_cast<const char*>(a.buffers[1]) + start * width, bytes, st));
    p->bufs[1] = p->owned[1];
  }
  CUDA_TRY(cudaStreamSynchronize(st));
  memset(out, 0, sizeof *out);
  out->array.length = n;
  out->array.null_count = has_nulls ? a.null_count : 0;
  out->array.offset = k;
  out->array.n_buffers = is_str ? 3 : 2;
  out->array.n_children = 0;
  out->array.buffers = p->bufs;
  out->array.release = dev_array_release;
  out->device_id = device;
  out->device_type = ARROW_DEVICE_CUDA;
  out->sync_event = nullptr;
  guard.p = nullptr;
  out->array.private_data = p.release();
  return PA_OK;
}

// ---- stable argsort of one column (sort.cuh): Series::sort / argsort, DataFrame::sort_index / sort_values ----
// The result lives on a pa_groupby handle in "sorted" state: its row order / inverse order are what a groupings build
// leaves there, so pa_groupby_take_grouped takes any column into sorted order with the scatter-shaped kernel.
}  // extern "C"
template <int VC>
static int sort_build_t(pa_groupby* g, const Column& col, bool descending) {
  cudaStream_t st = g->stream;
  const int64_t n = g->n;
  const size_t nb4 = static_cast<size_t>(std::max<int64_t>(n, 1)) * 4, nb8 = nb4 * 2;
  PA_TRY(g->grp_order.alloc(nb4, st));
  PA_TRY(g->grp_dest.alloc(nb4, st));
  if (n == 0) return PA_OK;
  DevBuf keys_a, keys_b, pay_a, pay_b, cls, hist, counts, tile_sums;
  PA_TRY(keys_a.alloc(nb8, st));
  PA_TRY(cls.alloc(static_cast<size_t>(n), st));
  PA_TRY(hist.alloc(sizeof(uint32_t) * (LS_DIGITS * CS_R + 4), st));
  CUDA_TRY(cudaMemsetAsync(hist.p, 0, sizeof(uint32_t) * (LS_DIGITS * CS_R + 4), st));
  SortKeyArgs ka{};
  ka.vals = col.data; ka.valid = col.valid; ka.voff = col.bit_off; ka.n = n; ka.vw = col.width; ka.descending = descending ? 1 : 0;
  ka.keys = keys_a.as<uint64_t>(); ka.cls = cls.as<uint8_t>(); ka.hist = hist.as<uint32_t>(); ka.flags = hist.as<uint32_t>() + LS_DIGITS * CS_R;
  const int kgrid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((n + 511) / 512, static_cast<int64_t>(g->num_sms) * 4)));
  k_sort_keys<VC><<<kgrid, 512, 0, st>>>(ka);
  CUDA_TRY(cudaGetLastError());
  std::vector<uint32_t> h(LS_DIGITS * CS_R + 4);
  CUDA_TRY(cudaMemcpyAsync(h.data(), hist.p, h.size() * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  // passes: every digit that is not constant over the column, then the class byte when NaNs / nulls exist
  std::vector<int> passes;
  for (int d = 0; d < LS_DIGITS; ++d) {
    bool constant = false;
    for (int b = 0; b < CS_R; ++b) if (h[d * CS_R + b] == static_cast<uint64_t>(n)) { constant = true; break; }
    if (!constant) passes.push_back(d);
  }
  if (h[LS_DIGITS * CS_R] & 1u) passes.push_back(-1);
  const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, static_cast<int64_t>(g->num_sms) * 16)));
  if (passes.empty()) {
    k_ls_identity<<<grid, 256, 0, st>>>(g->grp_order.as<uint32_t>(), g->grp_dest.as<uint32_t>(), n);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(st));
    return PA_OK;
  }
  const int64_t ntiles = (n + CS_TILE - 1) / CS_TILE;
  const int nb = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(ntiles, static_cast<int64_t>(g->num_sms) * 4)));
  const int64_t chunk = ((ntiles + nb - 1) / nb) * CS_TILE;
  PA_TRY(counts.alloc(sizeof(uint32_t) * CS_R * static_cast<size_t>(nb), st));
  if (passes.size() > 1) {
    PA_TRY(keys_b.alloc(nb8, st));
    PA_TRY(pay_a.alloc(nb4, st));
    if (passes.size() > 2) PA_TRY(pay_b.alloc(nb4, st));
  }
  CUDA_TRY(cudaFuncSetAttribute(k_ls_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(CS_SMEM)));
  const uint64_t* in_keys = keys_a.as<uint64_t>();
  const uint32_t* in_pay = nullptr;
  for (size_t p = 0; p < passes.size(); ++p) {
    const bool last = p + 1 == passes.size();
    LsArgs a{};
    a.keys = in_keys; a.payload = in_pay; a.n = n; a.nb = nb; a.chunk = chunk;
    a.cls = passes[p] < 0 ? cls.as<uint8_t>() : nullptr;
    a.shift = passes[p] < 0 ? 0 : passes[p] * CS_BITS;
    a.counts = counts.as<uint32_t>();
    DevBuf& ok = (p % 2 == 0) ? keys_b : keys_a;          // (keys_a holds the input of pass 0)
    DevBuf& op = (p % 2 == 0) ? pay_a : pay_b;
    a.out_keys = last ? nullptr : ok.as<uint64_t>();
    a.out_payload = last ? g->grp_order.as<uint32_t>() : op.as<uint32_t>();
    a.out_dest = last ? g->grp_dest.as<uint32_t>() : nullptr;
    k_ls_hist<<<nb, CS_THREADS, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    PA_TRY(scan_u32_on(g, counts.as<uint32_t>(), static_cast<uint64_t>(CS_R) * nb, &tile_sums));
    k_ls_scatter<<<nb, CS_THREADS, CS_SMEM, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    in_keys = a.out_keys;
    in_pay = a.out_payload;
  }
  CUDA_TRY(cudaStreamSynchronize(st));   // the ping-pong buffers are released here
  return PA_OK;
}
extern "C" {

int pa_sort_create(const struct ArrowDeviceArray* values, const struct ArrowSchema* schema, int32_t ascending,
                   const pa_options* opt, pa_groupby** out) {
  if (!values || !schema || !out) return set_err(PA_ERR_INVALID, "pa_sort_create: null argument");
  if (schema->dictionary) return set_err(PA_ERR_NOT_IMPLEMENTED, "sorting dictionary-encoded columns");
  HandlePtr g(new pa_groupby());
  PA_TRY(handle_init(g.get(), opt));
  cudaStream_t st = g->stream;
  g->keys.resize(1);
  Column& col = g->keys[0];
  PA_TRY(load_column(values, schema, st, g->device, &col));
  if (col.is_str || col.is_bool) return set_err(PA_ERR_NOT_IMPLEMENTED, "sorting '%s' columns (numeric and temporal types only)", schema->format);
  g->n = col.n;
  if (g->n >= (1ll << 31)) return set_err(PA_ERR_INVALID, "sort uses 32-bit row numbers: at most 2^31 - 1 rows");
  CUDA_TRY(cudaEventRecord(g->ev[6], st));
  int rc;
  if (col.vc == VC_F) rc = sort_build_t<VC_F>(g.get(), col, !ascending);
  else if (col.vc == VC_I) rc = sort_build_t<VC_I>(g.get(), col, !ascending);
  else rc = sort_build_t<VC_U>(g.get(), col, !ascending);
  PA_TRY(rc);
  CUDA_TRY(cudaEventRecord(g->ev[7], st));
  CUDA_TRY(cudaEventRecord(g->ev[8], st));
  CUDA_TRY(cudaEventRecord(g->ev[9], st));
  CUDA_TRY(cudaStreamSynchronize(st));
  g->sorted_state = true;
  g->have_groups = true;
  g->G = 0;
  g->have_groupings = true;
  *out = g.release();
  return PA_OK;
}

int pa_sort_indices(pa_groupby* g, struct ArrowArray* out, struct ArrowSchema* out_schema) {
  if (!g || !out || !out_schema) return set_err(PA_ERR_INVALID, "null argument");
  if (!g->sorted_state) return set_err(PA_ERR_STATE, "not a handle made by pa_sort_create");
  cudaStream_t st = g->stream;
  CUDA_TRY(cudaSetDevice(g->device));
  DevBuf wide;
  PA_TRY(wide.alloc(static_cast<size_t>(std::max<int64_t>(g->n, 1)) * 8, st));
  if (g->n > 0) {
    const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((g->n + 255) / 256, static_cast<int64_t>(g->num_sms) * 16)));
    k_ls_widen<<<grid, 256, 0, st>>>(g->grp_order.as<uint32_t>(), wide.as<uint64_t>(), g->n);
    CUDA_TRY(cudaGetLastError());
  }
  return export_host(st, "L", 8, static_cast<uint32_t>(g->n), wide.p, nullptr, out, out_schema);
}

// ---- multi-GPU partial export / merge ----
// A hashed composite key's word is a hash that an owner could only check against the key's columns, which do not
// travel: such a key groups on one GPU.
static int check_not_hashed_composite(const pa_groupby* g) {
  if (g->hashed && g->keys.size() > 1)
    return set_err(PA_ERR_NOT_IMPLEMENTED, "a hashed composite key (one wider than 64 bits, or with a utf8 column) groups on one GPU: "
                                           "it has no key layout, partial records or distinct pairs to exchange across shards or chunks");
  return PA_OK;
}

// keys the plain record exchange routes: one fixed-width column, a packed composite key or a resample index.  A utf8
// key's record carries a hash the owner cannot check without the key bytes: the _utf8 entry points export both.
static int check_shardable(const pa_groupby* g) {
  PA_TRY(check_not_hashed_composite(g));
  if (!g->resample && g->keys[0].is_str)
    return set_err(PA_ERR_NOT_IMPLEMENTED, "partial records of utf8 keys need their key bytes: use pa_groupby_partials_count_utf8 / "
                                           "pa_groupby_partials_export_utf8 (the padded exchange does not take utf8 keys)");
  return PA_OK;
}

static bool is_str_key(const pa_groupby* g) { return g->hashed && g->keys.size() == 1; }

static int check_composite_local(const pa_groupby* g) {
  PA_TRY(check_not_hashed_composite(g));
  if (g->resample || g->merged || !g->packed) return set_err(PA_ERR_INVALID, "key layouts describe the composite key (2+ columns) of a pa_groupby_create handle");
  return PA_OK;
}

// The current layout with its dictionary fingerprints
static int key_layout_of(pa_groupby* g, pa_key_layout* out) {
  PA_TRY(check_composite_local(g));
  fields_layout(g, out);
  return fill_fingerprints(g, out);
}

int pa_groupby_key_layout(pa_groupby* g, pa_key_layout* out) {
  if (!g || !out) return set_err(PA_ERR_INVALID, "null argument");
  return key_layout_of(g, out);
}

int pa_key_layout_agree(const pa_key_layout* all, int32_t n, pa_key_layout* out) {
  if (!all || !out || n < 1) return set_err(PA_ERR_INVALID, "bad argument (n >= 1 layouts)");
  for (int i = 0; i < n; ++i) PA_TRY(check_layout(all[i], i));
  pa_key_layout r = all[0];
  for (int i = 1; i < n; ++i) {
    const pa_key_layout& l = all[i];
    if (l.n_keys != r.n_keys) return set_err(PA_ERR_INVALID, "key layouts differ in their number of key columns (%d vs %d)", r.n_keys, l.n_keys);
    for (int j = 0; j < r.n_keys; ++j) {
      if (l.width[j] != r.width[j]) return set_err(PA_ERR_INVALID, "key column %d: widths differ across shards (%d vs %d bytes)", j, r.width[j], l.width[j]);
      // (before the bits: dictionaries of different lengths are a dictionary mismatch too)
      if (l.dict_fingerprint[j] != r.dict_fingerprint[j])
        return set_err(PA_ERR_INVALID, "key column %d: dictionaries differ across shards; encode the column against one dictionary shared by all shards", j);
      if (l.bits[j] != r.bits[j]) return set_err(PA_ERR_INVALID, "key column %d: value bits differ across shards (%d vs %d)", j, r.bits[j], l.bits[j]);
      r.nullable[j] |= l.nullable[j];
    }
  }
  std::vector<KeyField> fields;
  PA_TRY(layout_fields(r, &fields));
  *out = r;
  return PA_OK;
}

int pa_groupby_set_key_layout(pa_groupby* g, const pa_key_layout* layout) {
  if (!g || !layout) return set_err(PA_ERR_INVALID, "null argument");
  PA_TRY(check_composite_local(g));
  PA_TRY(check_layout(*layout, 0));
  PA_TRY(ensure_device(g));
  PA_TRY(finish_pending(g));
  pa_key_layout own;
  column_layout(g, &own);
  PA_TRY(fill_fingerprints(g, &own));
  if (layout->n_keys != own.n_keys) return set_err(PA_ERR_INVALID, "the layout has %d key columns, the handle %d", layout->n_keys, own.n_keys);
  for (int j = 0; j < own.n_keys; ++j) {
    if (layout->width[j] != own.width[j]) return set_err(PA_ERR_INVALID, "key column %d: the layout says %d bytes, the column has %d", j, layout->width[j], own.width[j]);
    if (layout->dict_fingerprint[j] != own.dict_fingerprint[j])
      return set_err(PA_ERR_INVALID, "key column %d: the layout's dictionary differs from the column's; encode the column against one dictionary shared by all shards", j);
    if (layout->bits[j] != own.bits[j]) return set_err(PA_ERR_INVALID, "key column %d: the layout says %d value bits, the column needs %d", j, layout->bits[j], own.bits[j]);
    if (own.nullable[j] && !layout->nullable[j]) return set_err(PA_ERR_INVALID, "key column %d has nulls, the layout gives it no null bit", j);
  }
  pa_key_layout cur;
  fields_layout(g, &cur);
  bool same = true;
  for (int j = 0; j < own.n_keys; ++j) same = same && cur.nullable[j] == layout->nullable[j];
  if (same) return PA_OK;
  std::vector<KeyField> fields;
  PA_TRY(layout_fields(*layout, &fields));
  g->fields = std::move(fields);
  PA_TRY(pack_keys(g));
  drop_results(g);
  return PA_OK;
}

int pa_merge_set_key_layout(pa_groupby* merged, const pa_key_layout* layout, const char* const* key_formats) {
  if (!merged || !layout || !key_formats) return set_err(PA_ERR_INVALID, "null argument");
  if (!merged->merged || merged->resample) return set_err(PA_ERR_STATE, "a merged key layout applies to a handle made by pa_merge_create / pa_merge_create_padded");
  if (!merged->packed && merged->keys[0].format != "L")
    return set_err(PA_ERR_INVALID, "composite keys travel as their packed word: merge with key format \"L\", not '%s'", merged->keys[0].format.c_str());
  PA_TRY(check_layout(*layout, 0));
  return set_merged_layout(merged, *layout, key_formats);
}

// The groups of the last aggregate and the values its records carry (records of any width)
static PartialsArgs partials_args(pa_groupby* g, int32_t n_parts) {
  PartialsArgs a{};
  a.r = g->res; a.G = g->G; a.nparts = n_parts; a.row_base = g->opt.row_base;
  a.vw = g->last_vw; a.wide = g->last_wide;
  for (auto& o : g->outs) {
    if (o.bit == AGG_FIRST) { a.first_vals = o.values.p; a.first_valid = o.valid.as<uint32_t>(); }
    if (o.bit == AGG_LAST) { a.last_vals = o.values.p; a.last_valid = o.valid.as<uint32_t>(); }
  }
  return a;
}

// Stream ordered: groups per owner added into d_counts[0 .. n_parts).
static int partials_count_async(pa_groupby* g, int32_t n_parts, unsigned long long* d_counts) {
  PartialsArgs a = partials_args(g, n_parts);
  a.counts = d_counts;
  if (g->G) {
    k_partials_count<<<(g->G + 255) / 256, 256, 0, g->stream>>>(a);
    CUDA_TRY(cudaGetLastError());
  }
  return PA_OK;
}

// counts_host[0 .. n_parts) = what `count_async` (partials_count_async, pairs_count_async) counts per owner.
static int owner_counts(pa_groupby* g, int32_t n_parts, int (*count_async)(pa_groupby*, int32_t, unsigned long long*), int64_t* counts_host) {
  cudaStream_t st = g->stream;
  DevBuf counts;
  PA_TRY(counts.alloc(sizeof(uint64_t) * n_parts, st));
  CUDA_TRY(cudaMemsetAsync(counts.p, 0, sizeof(uint64_t) * n_parts, st));
  PA_TRY(count_async(g, n_parts, counts.as<unsigned long long>()));
  std::vector<uint64_t> h(static_cast<size_t>(n_parts));
  CUDA_TRY(cudaMemcpyAsync(h.data(), counts.p, sizeof(uint64_t) * n_parts, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  for (int i = 0; i < n_parts; ++i) counts_host[i] = static_cast<int64_t>(h[i]);
  return PA_OK;
}

// Write cursors of a scatter grouped by owner: the exclusive prefix of the per-owner counts, copied to *cursor in stream
// order (from pageable memory: the copy has read `prefix` when it returns).
static int owner_cursors(cudaStream_t st, const int64_t* counts, int32_t n_parts, DevBuf* cursor) {
  std::vector<uint64_t> prefix(static_cast<size_t>(n_parts), 0);
  for (int i = 1; i < n_parts; ++i) prefix[i] = prefix[i - 1] + static_cast<uint64_t>(counts[i - 1]);
  PA_TRY(cursor->alloc(sizeof(uint64_t) * n_parts, st));
  CUDA_TRY(cudaMemcpyAsync(cursor->p, prefix.data(), sizeof(uint64_t) * n_parts, cudaMemcpyHostToDevice, st));
  return PA_OK;
}

int pa_groupby_partials_count(pa_groupby* g, int32_t n_parts, int64_t* counts_host) {
  if (!g || !counts_host || n_parts < 1 || n_parts > 64) return set_err(PA_ERR_INVALID, "bad argument (1 <= n_parts <= 64)");
  PA_TRY(finish_pending(g));
  if (!g->have_groups || g->merged) return set_err(PA_ERR_STATE, "partials need a finished local aggregate");
  PA_TRY(check_shardable(g));
  PA_TRY(ensure_device(g));
  PA_TRY(owner_counts(g, n_parts, partials_count_async, counts_host));
  g->parts_n = n_parts;
  g->parts_counts.assign(counts_host, counts_host + n_parts);
  return PA_OK;
}

static_assert(REC_WORDS == PA_PARTIAL_WORDS && REC_WORDS_STAGE2 == PA_PARTIAL_WORDS_STAGE2, "public record widths");

// `words`: REC_WORDS (the public record), REC_WORDS_STAGE2 (plus the stage-2 terms of the last aggregate) or
// REC_WORDS_COMPACT (merge.cuh) — the sharded step's own format for narrow aggregate sets
static int partials_export(pa_groupby* g, int32_t n_parts, void* dev_records, int64_t capacity_records, int words) {
  if (!g || !dev_records) return set_err(PA_ERR_INVALID, "null argument");
  if (g->parts_n != n_parts) return set_err(PA_ERR_STATE, "call pa_groupby_partials_count(n_parts=%d) first", n_parts);
  if (capacity_records < static_cast<int64_t>(g->G)) return set_err(PA_ERR_INVALID, "record buffer too small");
  PA_TRY(ensure_device(g));
  cudaStream_t st = g->stream;
  DevBuf cursor;
  PA_TRY(owner_cursors(st, g->parts_counts.data(), n_parts, &cursor));
  PartialsArgs a = partials_args(g, n_parts);
  a.words = words;
  if (words == REC_WORDS_STAGE2) {
    if (!g->s2_ext) return set_err(PA_ERR_STATE, "the last aggregate computed no product / variance / stddev: nothing for stage-2 records");
    // integer values: the merge recomputes the mean M2 was taken around from the double sum
    if (g->last_vc != VC_F && (g->s2_ext & (AGG_VARIANCE | AGG_STDDEV)) && !g->res.dsum)
      return set_err(PA_ERR_STATE, "stage-2 export: the last aggregate kept no double sum");
    a.m2 = (g->s2_ext & (AGG_VARIANCE | AGG_STDDEV)) ? g->s2_m2.as<double>() : nullptr;
    a.prod = (g->s2_ext & AGG_PRODUCT) ? g->s2_prod.as<unsigned long long>() : nullptr;
  }
  a.cursor = cursor.as<unsigned long long>();
  a.records = static_cast<uint64_t*>(dev_records);
  if (g->G) {
    k_partials_scatter<<<(g->G + 255) / 256, 256, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
  }
  CUDA_TRY(cudaStreamSynchronize(st));   // `cursor` dies here; records are complete for the caller's collective
  return PA_OK;
}

int pa_groupby_partials_export(pa_groupby* g, int32_t n_parts, void* dev_records, int64_t capacity_records) {
  if (g) PA_TRY(check_not_hashed_composite(g));
  return partials_export(g, n_parts, dev_records, capacity_records, REC_WORDS);
}

int pa_groupby_partials_export_stage2(pa_groupby* g, int32_t n_parts, void* dev_records, int64_t capacity_records) {
  if (g && g->merged) return set_err(PA_ERR_STATE, "partials need a finished local aggregate");
  if (g) PA_TRY(check_not_hashed_composite(g));
  return partials_export(g, n_parts, dev_records, capacity_records, REC_WORDS_STAGE2);
}

// ---- count_distinct across shards: distinct-pair records (distinct.cuh) ----
static_assert(DP_WORDS == PA_DISTINCT_PAIR_WORDS && DPF_KEY_NULL == 1, "public distinct-pair record");

static int pairs_check(pa_groupby* g, int32_t n_parts) {
  if (n_parts < 1 || n_parts > 64) return set_err(PA_ERR_INVALID, "bad argument (1 <= n_parts <= 64)");
  PA_TRY(finish_pending(g));
  if (g->merged) return set_err(PA_ERR_STATE, "distinct pairs come from a local aggregate, not from a merged handle");
  PA_TRY(check_not_hashed_composite(g));
  if (!g->cd_have) return set_err(PA_ERR_STATE, "the last aggregate computed no count_distinct: no distinct pairs to export");
  return ensure_device(g);
}

static PairsArgs pairs_args(pa_groupby* g, int32_t n_parts) {
  PairsArgs a{};
  a.r = g->res;
  a.id = g->cd_id.as<uint32_t>();
  a.bits = g->cd_bits.as<uint64_t>();
  a.n = g->cd_n;
  a.nparts = static_cast<uint32_t>(n_parts);
  return a;
}

// Stream ordered: pairs per owner added into d_counts[0 .. n_parts).
static int pairs_count_async(pa_groupby* g, int32_t n_parts, unsigned long long* d_counts) {
  PairsArgs a = pairs_args(g, n_parts);
  a.counts = d_counts;
  if (a.n) {
    k_pairs_count<<<static_cast<unsigned>((a.n + 255) / 256), 256, 0, g->stream>>>(a);
    CUDA_TRY(cudaGetLastError());
  }
  return PA_OK;
}

// The pairs grouped by owner (counts per owner as pa_groupby_distinct_pairs_count gave them); complete on return.
static int pairs_export(pa_groupby* g, int32_t n_parts, const int64_t* counts, void* dev_pairs, DevBuf* d_cursor) {
  cudaStream_t st = g->stream;
  PA_TRY(owner_cursors(st, counts, n_parts, d_cursor));
  PairsArgs a = pairs_args(g, n_parts);
  a.cursor = d_cursor->as<unsigned long long>();
  a.out = static_cast<uint64_t*>(dev_pairs);
  if (a.n) {
    k_pairs_scatter<<<static_cast<unsigned>((a.n + 255) / 256), 256, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
  }
  CUDA_TRY(cudaStreamSynchronize(st));
  return PA_OK;
}

int pa_groupby_distinct_pairs_count(pa_groupby* g, int32_t n_parts, int64_t* counts_host) {
  if (!g || !counts_host) return set_err(PA_ERR_INVALID, "null argument");
  PA_TRY(pairs_check(g, n_parts));
  PA_TRY(owner_counts(g, n_parts, pairs_count_async, counts_host));
  g->dp_parts_n = n_parts;
  g->dp_counts.assign(counts_host, counts_host + n_parts);
  return PA_OK;
}

int pa_groupby_distinct_pairs_export(pa_groupby* g, int32_t n_parts, void* dev_pairs, int64_t capacity_pairs) {
  if (!g || !dev_pairs) return set_err(PA_ERR_INVALID, "null argument");
  PA_TRY(pairs_check(g, n_parts));
  if (g->dp_parts_n != n_parts) return set_err(PA_ERR_STATE, "call pa_groupby_distinct_pairs_count(n_parts=%d) first", n_parts);
  if (capacity_pairs < 0 || static_cast<uint64_t>(capacity_pairs) < g->cd_n) return set_err(PA_ERR_INVALID, "pair buffer too small");
  DevBuf cursor;
  return pairs_export(g, n_parts, g->dp_counts.data(), dev_pairs, &cursor);
}

int pa_merge_create(const void* dev_records, const int64_t* counts_by_source, int32_t n_sources, uint32_t agg_mask,
                    const char* value_format, const char* key_format, const pa_options* opt, pa_groupby** out) {
  if (!counts_by_source || n_sources < 1 || !value_format || !key_format || !out) return set_err(PA_ERR_INVALID, "null argument");
  // (count_distinct does not travel in partial records: pa_merge_distinct_pairs adds it to the merged handle)
  if (agg_mask & ~RECORD_AGGS) return set_err(PA_ERR_INVALID, "bad aggregate mask");
  if ((agg_mask & (PA_AGG_BOOL_ALL | PA_AGG_BOOL_ANY)) && strcmp(value_format, "b") != 0)
    return set_err(PA_ERR_INVALID, "all / any need a boolean column (arrow::compute has no kernel for other types)");
  HandlePtr g(new pa_groupby());
  PA_TRY(handle_init(g.get(), opt));
  for (int i = 0; i < n_sources; ++i)
    if (counts_by_source[i] < 0) return set_err(PA_ERR_INVALID, "negative record count");
  PA_TRY(merge_counted(g.get(), dev_records, counts_by_source, n_sources, agg_mask, value_format, key_format, nullptr, 0, false));
  if (g->ks_str) {   // (pa_merge_key_strings maps these records to their groups; the caller keeps them alive until then)
    g->ks_recs = dev_records;
    g->ks_words = record_words(agg_mask, false);
    g->ks_nrec = 0;
    for (int i = 0; i < n_sources; ++i) g->ks_nrec += static_cast<uint64_t>(counts_by_source[i]);
  }
  *out = g.release();
  return PA_OK;
}

// Owner-side count_distinct of a merged handle from n_pairs received distinct-pair records (any order): every pair is
// mapped to its merged group through the key lookup table of build_row_lookup, inserted into a set of (bits, group) of
// 2^k >= 2 n_pairs 16-byte slots (kept in *keep between calls when given), and counted when it was new.  Replaces an
// earlier PA_AGG_COUNT_DISTINCT output.  `set_slots`: the set's size.
static int merge_distinct(pa_groupby* g, const void* dev_pairs, uint64_t n_pairs, DevBuf* keep, uint64_t* set_slots) {
  cudaStream_t st = g->stream;
  const uint32_t G = g->G;
  keep_outputs(g, ~PA_AGG_COUNT_DISTINCT);
  uint64_t cap = 1024;
  while (cap < 2 * n_pairs) cap <<= 1;
  DevBuf local_set, distinct, flag;
  DevBuf& set = keep ? *keep : local_set;
  PA_TRY(distinct.alloc(static_cast<size_t>(std::max<uint32_t>(G, 1)) * 8, st));
  CUDA_TRY(cudaMemsetAsync(distinct.p, 0, static_cast<size_t>(std::max<uint32_t>(G, 1)) * 8, st));
  PA_TRY(flag.alloc(4, st));
  CUDA_TRY(cudaMemsetAsync(flag.p, 0, 4, st));
  RowLookup lk;
  if (n_pairs) {
    PA_TRY(set.alloc(cap * sizeof(DistinctSlot), st));
    CUDA_TRY(cudaMemsetAsync(set.p, 0xFF, cap * sizeof(DistinctSlot), st));
    PA_TRY(build_row_lookup(g, &lk));
    DistinctMergeArgs a{};
    a.ids = lk.a;
    a.pairs = static_cast<const uint64_t*>(dev_pairs);
    a.n = n_pairs;
    a.set = set.as<DistinctSlot>();
    a.cap_mask = cap - 1;
    a.distinct = distinct.as<unsigned long long>();
    a.G = G;
    a.no_group = flag.as<uint32_t>();
    const int grid = static_cast<int>(std::min<uint64_t>((n_pairs + DM_THREADS - 1) / DM_THREADS, static_cast<uint64_t>(g->num_sms) * 8));
    if (G <= DM_SMEM_GROUPS) k_distinct_merge<true><<<grid, DM_THREADS, static_cast<size_t>(std::max<uint32_t>(G, 1)) * 4, st>>>(a);
    else k_distinct_merge<false><<<grid, DM_THREADS, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
  }
  g->outs.emplace_back();
  AggOut& o = g->outs.back();
  o.bit = PA_AGG_COUNT_DISTINCT;
  o.format = "l";
  o.width = 8;
  o.nullable = false;
  PA_TRY(o.values.alloc(static_cast<size_t>(std::max<uint32_t>(G, 1)) * 8, st));
  if (G) {
    k_distinct_emit<<<(G + 255) / 256, 256, 0, st>>>(distinct.as<unsigned long long>(), G, o.values.as<int64_t>());
    CUDA_TRY(cudaGetLastError());
  }
  uint32_t h_flag = 0;
  CUDA_TRY(cudaMemcpyAsync(&h_flag, flag.p, 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));   // the lookup table and the local set are released after this point
  if (set_slots) *set_slots = n_pairs ? cap : 0;
  if (h_flag) {
    g->outs.pop_back();
    return set_err(PA_ERR_STATE, "a distinct pair names a key that no merged record carried (inconsistent exchange)");
  }
  return PA_OK;
}

int pa_merge_distinct_pairs(pa_groupby* merged, const void* dev_pairs, const int64_t* counts_by_source, int32_t n_sources) {
  if (!merged || !counts_by_source || n_sources < 1) return set_err(PA_ERR_INVALID, "null argument");
  PA_TRY(finish_pending(merged));
  if (!merged->merged || !merged->have_groups) return set_err(PA_ERR_STATE, "distinct pairs merge into a handle made by pa_merge_create");
  if (merged->ks_str && !merged->ks_have)
    return set_err(PA_ERR_STATE, "utf8 merged handle: attach the key strings with pa_merge_key_strings before merging distinct pairs");
  uint64_t total = 0;
  for (int i = 0; i < n_sources; ++i) {
    if (counts_by_source[i] < 0) return set_err(PA_ERR_INVALID, "negative pair count");
    total += static_cast<uint64_t>(counts_by_source[i]);
  }
  if (total > 0xFFFFFFFEull) return set_err(PA_ERR_INVALID, "more than 2^32 - 2 distinct pairs in one merge");
  if (total && !dev_pairs) return set_err(PA_ERR_INVALID, "null pair buffer");
  PA_TRY(ensure_device(merged));
  return merge_distinct(merged, dev_pairs, total, nullptr, nullptr);
}

// ---- utf8 keys across shards: the key bytes travel with the records (strkeys.cuh) ----
// In-place exclusive scan of n 64-bit words (cub); `tmp`: its scratch
static int scan_u64(cudaStream_t st, unsigned long long* data, uint64_t n, DevBuf* tmp) {
  size_t bytes = 0;
  CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, bytes, data, static_cast<int64_t>(n), st));
  PA_TRY(tmp->alloc(std::max<size_t>(bytes, 1), st));
  CUDA_TRY(cub::DeviceScan::ExclusiveSum(tmp->p, bytes, data, static_cast<int64_t>(n), st));
  return PA_OK;
}

// Stream ordered: key bytes per owner of the G local groups (GroupResult, or the unordered bucket records when
// `unordered_recs` is given) added into d_bytes[0 .. n_parts)
static int keystr_count_async(pa_groupby* g, int32_t n_parts, const void* unordered_recs, uint32_t G, unsigned long long* d_bytes) {
  if (!G) return PA_OK;
  if (unordered_recs)
    k_keystr_count_bk<<<(G + 255) / 256, 256, 0, g->stream>>>(g->keys[0].str, static_cast<const BkRec32*>(unordered_recs), G, static_cast<uint32_t>(n_parts), d_bytes);
  else
    k_keystr_count<<<(G + 255) / 256, 256, 0, g->stream>>>(g->keys[0].str, g->res, G, static_cast<uint32_t>(n_parts), d_bytes);
  CUDA_TRY(cudaGetLastError());
  return PA_OK;
}

// Lengths and key bytes of n exported records (`words` wide, in the order they were written): lengths[i], and the bytes
// at the exclusive prefix of the lengths — owner segments are contiguous, so the bytes are grouped by owner too.
// `off`, `tmp`: scratch.  Stream ordered.
static int keystr_export(pa_groupby* g, const uint64_t* recs, int words, uint64_t n, uint32_t* lengths, uint8_t* bytes, DevBuf* off, DevBuf* tmp) {
  cudaStream_t st = g->stream;
  PA_TRY(off->alloc((n + 1) * 8, st));
  k_keystr_lengths<<<static_cast<unsigned>((n + 1 + 255) / 256), 256, 0, st>>>(g->keys[0].str, recs, words, n, g->opt.row_base, lengths,
                                                                                off->as<unsigned long long>());
  CUDA_TRY(cudaGetLastError());
  PA_TRY(scan_u64(st, off->as<unsigned long long>(), n + 1, tmp));
  if (n) {
    k_keystr_pack<<<static_cast<unsigned>((n * 32 + 255) / 256), 256, 0, st>>>(g->keys[0].str, recs, words, n, g->opt.row_base,
                                                                               off->as<unsigned long long>(), bytes);
    CUDA_TRY(cudaGetLastError());
  }
  return PA_OK;
}

// Owner side, after the record merge: the received records (`words` wide, nrec, as merged) with their lengths and key
// bytes -> merged group and representative of every record, byte check against the representative.  Attaches the G
// representative strings, compacted, to m — unless two different strings share a merged group: then *collided and
// nothing is attached (the ranks retry with the next hash seed).  `bytes_expected`: what the sources say they sent.
static int merge_key_strings(pa_groupby* m, const uint64_t* recs, int words, uint64_t nrec, const uint32_t* lengths, const uint8_t* bytes,
                             uint64_t bytes_expected, bool* collided) {
  cudaStream_t st = m->stream;
  const uint32_t G = m->G;
  *collided = false;
  m->ks_have = false;
  DevBuf off, tmp, rec_group, rep, flag, out_off;
  PA_TRY(off.alloc((nrec + 1) * 8, st));
  k_keystr_widen<<<static_cast<unsigned>((nrec + 1 + 255) / 256), 256, 0, st>>>(lengths, nrec, off.as<unsigned long long>());
  CUDA_TRY(cudaGetLastError());
  PA_TRY(scan_u64(st, off.as<unsigned long long>(), nrec + 1, &tmp));
  PA_TRY(flag.alloc(4, st));
  CUDA_TRY(cudaMemsetAsync(flag.p, 0, 4, st));
  PA_TRY(rep.alloc(static_cast<size_t>(std::max<uint32_t>(G, 1)) * 4, st));
  CUDA_TRY(cudaMemsetAsync(rep.p, 0xFF, static_cast<size_t>(std::max<uint32_t>(G, 1)) * 4, st));
  PA_TRY(out_off.alloc((static_cast<size_t>(G) + 1) * 8, st));
  RowLookup lk;
  if (nrec) {
    PA_TRY(build_row_lookup(m, &lk));
    PA_TRY(rec_group.alloc(nrec * 4, st));
    k_keystr_rep<<<static_cast<unsigned>((nrec + 255) / 256), 256, 0, st>>>(recs, words, nrec, lk.a, m->m_first_row_g.as<uint64_t>(),
                                                                           rec_group.as<uint32_t>(), rep.as<uint32_t>(), flag.as<uint32_t>());
    CUDA_TRY(cudaGetLastError());
    k_keystr_verify<<<static_cast<unsigned>((nrec * 32 + 255) / 256), 256, 0, st>>>(recs, words, nrec, rec_group.as<uint32_t>(), rep.as<uint32_t>(),
                                                                                    off.as<unsigned long long>(), bytes, G, flag.as<uint32_t>());
    CUDA_TRY(cudaGetLastError());
  }
  k_keystr_rep_lengths<<<(G + 1 + 255) / 256, 256, 0, st>>>(rep.as<uint32_t>(), m->res.key_kind, G, off.as<unsigned long long>(),
                                                            out_off.as<unsigned long long>(), flag.as<uint32_t>());
  CUDA_TRY(cudaGetLastError());
  PA_TRY(scan_u64(st, out_off.as<unsigned long long>(), static_cast<uint64_t>(G) + 1, &tmp));
  uint32_t h_flag = 0;
  uint64_t h_total[2] = {0, 0};
  CUDA_TRY(cudaMemcpyAsync(&h_flag, flag.p, 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(&h_total[0], off.as<uint64_t>() + nrec, 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(&h_total[1], out_off.as<uint64_t>() + G, 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  if (h_total[0] != bytes_expected)
    return set_err(PA_ERR_INVALID, "the key-string lengths add up to %llu bytes, the sources sent %llu", (unsigned long long)h_total[0],
                   (unsigned long long)bytes_expected);
  if (h_flag & KS_NO_GROUP)
    return set_err(PA_ERR_STATE, "key strings do not match the merged records (a record names no merged group, or a group has no representative)");
  if (h_flag & KS_COLLISION) {
    *collided = true;
    return PA_OK;
  }
  PA_TRY(m->ks_bytes.alloc(std::max<uint64_t>(h_total[1], 1), st));
  PA_TRY(m->ks_rows.alloc(static_cast<size_t>(std::max<uint32_t>(G, 1)) * 4, st));
  if (G) {
    k_keystr_rep_gather<<<static_cast<unsigned>((static_cast<uint64_t>(G) * 32 + 255) / 256), 256, 0, st>>>(
        rep.as<uint32_t>(), G, off.as<unsigned long long>(), bytes, out_off.as<unsigned long long>(), m->ks_bytes.as<uint8_t>());
    CUDA_TRY(cudaGetLastError());
    k_iota_u32<<<(G + 255) / 256, 256, 0, st>>>(m->ks_rows.as<uint32_t>(), G);
    CUDA_TRY(cudaGetLastError());
  }
  m->ks_off = std::move(out_off);
  CUDA_TRY(cudaStreamSynchronize(st));   // the caller's record / byte buffers are read by now
  m->ks_have = true;
  return PA_OK;
}

int pa_groupby_key_hash_seed(pa_groupby* g, uint64_t* seed) {
  if (!g || !seed) return set_err(PA_ERR_INVALID, "null argument");
  if (!g->hashed)
    return set_err(PA_ERR_INVALID, "key hash seeds belong to a pa_groupby_create handle with a hashed key (one utf8 / large_utf8 key, "
                                   "or a composite key that does not pack into 64 bits)");
  *seed = g->key_seed;
  return PA_OK;
}

int pa_groupby_set_key_hash_seed(pa_groupby* g, uint64_t seed) {
  if (!g) return set_err(PA_ERR_INVALID, "null argument");
  if (!is_str_key(g)) return set_err(PA_ERR_INVALID, "key hash seeds belong to a pa_groupby_create handle with one utf8 / large_utf8 key");
  PA_TRY(ensure_device(g));
  PA_TRY(finish_pending(g));
  return set_key_seed(g, seed);
}

int pa_groupby_partials_count_utf8(pa_groupby* g, int32_t n_parts, int64_t* records_host, int64_t* bytes_host) {
  if (!g || !records_host || !bytes_host || n_parts < 1 || n_parts > 64) return set_err(PA_ERR_INVALID, "bad argument (1 <= n_parts <= 64)");
  PA_TRY(finish_pending(g));
  if (!g->have_groups || g->merged) return set_err(PA_ERR_STATE, "partials need a finished local aggregate");
  PA_TRY(check_not_hashed_composite(g));
  if (!is_str_key(g)) return set_err(PA_ERR_INVALID, "pa_groupby_partials_count_utf8 takes one utf8 / large_utf8 key; use pa_groupby_partials_count");
  PA_TRY(ensure_device(g));
  cudaStream_t st = g->stream;
  DevBuf counts;
  PA_TRY(counts.alloc(sizeof(uint64_t) * 2 * n_parts, st));
  CUDA_TRY(cudaMemsetAsync(counts.p, 0, sizeof(uint64_t) * 2 * n_parts, st));
  PA_TRY(partials_count_async(g, n_parts, counts.as<unsigned long long>()));
  PA_TRY(keystr_count_async(g, n_parts, nullptr, g->G, counts.as<unsigned long long>() + n_parts));
  std::vector<uint64_t> h(static_cast<size_t>(2 * n_parts));
  CUDA_TRY(cudaMemcpyAsync(h.data(), counts.p, sizeof(uint64_t) * 2 * n_parts, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  for (int i = 0; i < n_parts; ++i) {
    records_host[i] = static_cast<int64_t>(h[i]);
    bytes_host[i] = static_cast<int64_t>(h[n_parts + i]);
  }
  g->parts_n = n_parts;
  g->parts_counts.assign(records_host, records_host + n_parts);
  g->ks_counts.assign(bytes_host, bytes_host + n_parts);
  return PA_OK;
}

int pa_groupby_partials_export_utf8(pa_groupby* g, int32_t n_parts, int32_t stage2, void* dev_records, int64_t capacity_records,
                                    void* dev_lengths, void* dev_bytes, int64_t capacity_bytes) {
  if (!g || !dev_records) return set_err(PA_ERR_INVALID, "null argument");
  if (g->merged) return set_err(PA_ERR_STATE, "partials need a finished local aggregate");
  PA_TRY(check_not_hashed_composite(g));
  if (!is_str_key(g)) return set_err(PA_ERR_INVALID, "pa_groupby_partials_export_utf8 takes one utf8 / large_utf8 key; use pa_groupby_partials_export");
  if (g->parts_n != n_parts || g->ks_counts.size() != static_cast<size_t>(n_parts))
    return set_err(PA_ERR_STATE, "call pa_groupby_partials_count_utf8(n_parts=%d) first", n_parts);
  int64_t total = 0;
  for (int64_t b : g->ks_counts) total += b;
  if (capacity_bytes < total) return set_err(PA_ERR_INVALID, "key byte buffer too small (%lld bytes, %lld needed)", (long long)capacity_bytes, (long long)total);
  if ((g->G && !dev_lengths) || (total && !dev_bytes)) return set_err(PA_ERR_INVALID, "null length / byte buffer");
  const int words = stage2 ? REC_WORDS_STAGE2 : REC_WORDS;
  PA_TRY(partials_export(g, n_parts, dev_records, capacity_records, words));
  DevBuf off, tmp;
  PA_TRY(keystr_export(g, static_cast<const uint64_t*>(dev_records), words, g->G, static_cast<uint32_t*>(dev_lengths), static_cast<uint8_t*>(dev_bytes),
                       &off, &tmp));
  CUDA_TRY(cudaStreamSynchronize(g->stream));
  return PA_OK;
}

int pa_merge_key_strings(pa_groupby* merged, const void* dev_lengths, const void* dev_bytes, const int64_t* records_by_source,
                         const int64_t* bytes_by_source, const uint64_t* seed_by_source, int32_t n_sources, int32_t* collided) {
  if (!merged || !records_by_source || !bytes_by_source || !seed_by_source || n_sources < 1 || !collided) return set_err(PA_ERR_INVALID, "null argument");
  *collided = 0;
  PA_TRY(finish_pending(merged));
  if (!merged->merged || !merged->ks_str || !merged->have_groups)
    return set_err(PA_ERR_STATE, "key strings attach to a handle made by pa_merge_create with key format \"u\" / \"U\"");
  uint64_t nrec = 0, nbytes = 0;
  for (int i = 0; i < n_sources; ++i) {
    if (records_by_source[i] < 0 || bytes_by_source[i] < 0) return set_err(PA_ERR_INVALID, "negative record / byte count");
    nrec += static_cast<uint64_t>(records_by_source[i]);
    nbytes += static_cast<uint64_t>(bytes_by_source[i]);
    // differing hashes of one string merge into two groups, which no check after the merge can see
    if (seed_by_source[i] != seed_by_source[0])
      return set_err(PA_ERR_INVALID, "sources %d and 0 hashed their keys with different seeds (%llu vs %llu): agree on one seed "
                                     "(pa_groupby_set_key_hash_seed), aggregate again and redo the exchange", i,
                     (unsigned long long)seed_by_source[i], (unsigned long long)seed_by_source[0]);
  }
  if (nrec != merged->ks_nrec)
    return set_err(PA_ERR_INVALID, "records_by_source adds up to %llu records, pa_merge_create merged %llu", (unsigned long long)nrec,
                   (unsigned long long)merged->ks_nrec);
  if ((nrec && !dev_lengths) || (nbytes && !dev_bytes)) return set_err(PA_ERR_INVALID, "null length / byte buffer");
  PA_TRY(ensure_device(merged));
  bool c = false;
  PA_TRY(merge_key_strings(merged, static_cast<const uint64_t*>(merged->ks_recs), merged->ks_words, nrec, static_cast<const uint32_t*>(dev_lengths),
                           static_cast<const uint8_t*>(dev_bytes), nbytes, &c));
  *collided = c ? 1 : 0;
  return PA_OK;
}

int pa_groupby_partials_export_padded(pa_groupby* g, int32_t n_parts, void* dev_blocks, int64_t block_records) {
  if (!g || !dev_blocks || n_parts < 1 || n_parts > 64 || block_records < 1) return set_err(PA_ERR_INVALID, "bad argument (1 <= n_parts <= 64)");
  if (!g->have_groups || g->merged) return set_err(PA_ERR_STATE, "partials need a finished local aggregate");
  PA_TRY(check_shardable(g));
  PA_TRY(ensure_device(g));
  PartialsArgs a = partials_args(g, n_parts);
  a.words = REC_WORDS;
  a.records = static_cast<uint64_t*>(dev_blocks);
  if (g->pending) {   // deferred local aggregate: group count and failure flag are still on the device
    a.G_dev = g->status.as<uint32_t>() + ST_NGROUPS;
    a.abort_dev = g->status.as<uint32_t>() + ST_ABORT;
  }
  k_partials_pack_padded<<<1, 1024, 0, g->stream>>>(a, static_cast<uint64_t>(block_records));
  CUDA_TRY(cudaGetLastError());
  return PA_OK;   // stream ordered: no host synchronisation
}

int pa_merge_create_padded(const void* dev_blocks, int32_t n_sources, int64_t block_records, uint32_t agg_mask,
                           const char* value_format, const char* key_format, const pa_options* opt, pa_groupby** out) {
  if (!dev_blocks || n_sources < 1 || n_sources > 64 || block_records < 1 || !value_format || !key_format || !out)
    return set_err(PA_ERR_INVALID, "bad argument (1 <= n_sources <= 64)");
  if (agg_mask & ~PA_AGG_ALL) return set_err(PA_ERR_INVALID, "bad aggregate mask");
  if ((key_format[0] == 'u' || key_format[0] == 'U') && key_format[1] == 0)
    return set_err(PA_ERR_NOT_IMPLEMENTED, "utf8 keys take the counted exchange (pa_merge_create + pa_merge_key_strings), not padded blocks");
  HandlePtr g;
  {
    int dev = opt && opt->device >= 0 ? opt->device : -1;
    if (dev < 0) CUDA_TRY(cudaGetDevice(&dev));
    pa_groupby* recycled = (opt && opt->cuda_stream) ? pool_take(dev, static_cast<cudaStream_t>(opt->cuda_stream)) : nullptr;
    if (recycled) {
      g.reset(recycled);
      g->opt = *opt;
      CUDA_TRY(cudaSetDevice(g->device));
    } else {
      g.reset(new pa_groupby());
      PA_TRY(handle_init(g.get(), opt));
    }
  }
  g->poolable = false;
  cudaStream_t st = g->stream;
  const uint64_t nrec_max = static_cast<uint64_t>(n_sources) * static_cast<uint64_t>(block_records);
  CUDA_TRY(cudaMemsetAsync(g->status.p, 0, sizeof(uint32_t) * ST_WORDS, st));
  CUDA_TRY(cudaEventRecord(g->ev[0], st));
  // ---- few records: the whole merge is one single-CTA kernel + emit, one synchronisation ----
  PA_TRY(set_merged_formats(g.get(), value_format, key_format));
  g->last_wide = is_wide(agg_mask, g->last_vc);
  const uint32_t cap_out = static_cast<uint32_t>(std::min<uint64_t>(nrec_max, MS_MAX_GROUPS)) + 2;
  MergeSmallArgs m{};
  PA_TRY(alloc_merged_result(g.get(), cap_out, &m));
  m.blocks = static_cast<const uint64_t*>(dev_blocks);
  m.nsrc = static_cast<uint32_t>(n_sources);
  m.block_records = static_cast<uint64_t>(block_records);
  m.vc = g->last_vc;
  m.status = g->status.as<uint32_t>();
  static bool attr_set[64] = {};
  if (!attr_set[g->device & 63]) {
    CUDA_TRY(cudaFuncSetAttribute(k_merge_small, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(MS_SMEM_BYTES)));
    attr_set[g->device & 63] = true;
  }
  CUDA_TRY(cudaEventRecord(g->ev[1], st));
  k_merge_small<<<1, MS_THREADS, MS_SMEM_BYTES, st>>>(m);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaEventRecord(g->ev[2], st));
  CUDA_TRY(cudaEventRecord(g->ev[3], st));
  g->have_groups = true;
  g->last_launches = 1;
  g->last_path = 4;
  g->G = cap_out;                                     // upper bound for the emit grid and the output buffers
  g->emit_G_dev = g->status.as<uint32_t>() + ST_COUNTER;
  PA_TRY(run_emit(g.get(), nullptr, agg_mask));
  g->emit_G_dev = nullptr;
  CUDA_TRY(cudaEventRecord(g->ev[4], st));
  // the status words (group count, overflow markers) are read by the first call that needs them
  g->pending_merge = true;
  g->poolable = true;
  g->pm_blocks = dev_blocks; g->pm_nsrc = n_sources; g->pm_block_records = block_records; g->pm_mask = agg_mask;
  g->pm_vfmt = value_format; g->pm_kfmt = key_format;
  *out = g.release();
  return PA_OK;
}

// ---- host frames larger than the device (or than 2^32-2 rows): aggregate chunk by chunk, merge the partials ----
// The row-range shards of the multi-GPU path, executed one after the other on ONE device: every chunk of the host
// columns is copied (staged, §h2d_copy), aggregated with row_base = its first row, and exported as partial records;
// the owner-side merge then joins the chunks' records exactly as it joins ranks' — sources folded in chunk (= row)
// order, groups ordered by global first row.  Device memory in use: one chunk of keys and values + the records.
// Product / variance / stddev: every chunk's two-pass terms travel in stage-2 records (merge.cuh).  All / any: in the
// min / max words of the ordinary record.
int pa_groupby_aggregate_chunked(const struct ArrowDeviceArray* keys, const struct ArrowSchema* key_schema,
                                 const struct ArrowDeviceArray* values, const struct ArrowSchema* value_schema,
                                 uint32_t agg_mask, int64_t chunk_rows, const pa_options* opt, pa_groupby** merged_out) {
  return pa_groupby_aggregate_chunked_keys(keys, key_schema, 1, values, value_schema, agg_mask, chunk_rows, opt, merged_out);
}

// Composite keys: every chunk is a view of the same columns (same dictionaries, and a chunk of a column with nulls keeps
// the bitmap), so each chunk packs with the layout of the whole columns; that layout goes to the merged handle.
int pa_groupby_aggregate_chunked_keys(const struct ArrowDeviceArray* keys, const struct ArrowSchema* key_schemas, int32_t n_keys,
                                      const struct ArrowDeviceArray* values, const struct ArrowSchema* value_schema,
                                      uint32_t agg_mask, int64_t chunk_rows, const pa_options* opt, pa_groupby** merged_out) {
  if (!keys || !key_schemas || n_keys < 1 || !values || !value_schema || !merged_out) return set_err(PA_ERR_INVALID, "null argument");
  if (agg_mask == 0 || (agg_mask & ~RECORD_AGGS))
    return set_err(PA_ERR_NOT_IMPLEMENTED, "chunked aggregates: sum / mean / count / min / max / first / last / product / variance / stddev / "
                                           "all / any (count_distinct is not available across chunks)");
  const int RW = record_words(agg_mask, false);
  for (int j = 0; j < n_keys; ++j)
    if (keys[j].device_type == ARROW_DEVICE_CUDA || values->device_type == ARROW_DEVICE_CUDA)
      return set_err(PA_ERR_INVALID, "chunked aggregation is for HOST columns (device columns already fit the device)");
  const int64_t n = keys->array.length;
  if (values->array.length != n) return set_err(PA_ERR_INVALID, "key and value columns differ in length");
  for (int j = 1; j < n_keys; ++j)
    if (keys[j].array.length != n) return set_err(PA_ERR_INVALID, "key columns differ in length");
  const bool composite = n_keys > 1;
  pa_key_layout whole{};   // composite: the layout of the whole columns (as load_column + column_layout see them)
  if (composite && n_keys <= PA_MAX_KEY_COLS) {
    whole.n_keys = n_keys;
    for (int j = 0; j < n_keys; ++j) {
      int w = 8, vc = VC_I;
      if (parse_format(key_schemas[j].format, &w, &vc) != PA_OK) break;   // (pa_groupby_create reports it)
      whole.width[j] = w;
      whole.bits[j] = key_bits(w, key_schemas[j].dictionary != nullptr, keys[j].array.dictionary ? keys[j].array.dictionary->length : 0);
      whole.nullable[j] = keys[j].array.null_count != 0 && keys[j].array.buffers[0] != nullptr;
    }
  }
  if (chunk_rows <= 0) chunk_rows = 1ll << 30;
  if (chunk_rows >= 0xFFFFFFFEll) return set_err(PA_ERR_INVALID, "chunk_rows must be below 2^32 - 2");
  const int64_t n_chunks = std::max<int64_t>(1, (n + chunk_rows - 1) / chunk_rows);
  if (n_chunks > 64) return set_err(PA_ERR_INVALID, "%lld chunks: at most 64 (raise chunk_rows)", (long long)n_chunks);
  pa_options o;
  if (opt) o = *opt; else pa_options_init(&o);
  const int64_t base0 = o.row_base;
  // Chunks merge by their packed key words, so a composite key must pack into 64 bits — decided here, from the whole
  // columns, because pa_groupby_create would hash a chunk that does not pack
  if (composite) {
    for (int j = 0; j < n_keys; ++j) {
      const char* f = key_schemas[j].format;
      if (f && (f[0] == 'u' || f[0] == 'U') && f[1] == 0)
        return set_err(PA_ERR_NOT_IMPLEMENTED, "utf8 keys inside a composite key: dictionary-encode that column");
    }
    if (n_keys <= PA_MAX_KEY_COLS) {
      std::vector<KeyField> fields;
      PA_TRY(layout_fields(whole, &fields));
    }
  }
  // utf8 key: every chunk hashes with one seed and exports its key bytes next to its records; a chunk whose own check
  // moves the seed, or a merge that finds two strings under one hash, redoes the chunks with the next seed (four at most)
  const char* kf0 = key_schemas[0].format;
  const bool str = n_keys == 1 && kf0 && (kf0[0] == 'u' || kf0[0] == 'U') && kf0[1] == 0;
  for (uint64_t seed = 0;;) {
  if (seed >= 4) return set_err(PA_ERR_STATE, "utf8 keys: four differently seeded 64-bit hashes all collided");
  DevBuf records, lengths, bytes;      // all chunks' records (and key lengths / bytes), chunk after chunk
  records.plain = true; lengths.plain = true; bytes.plain = true;
  std::vector<int64_t> counts(static_cast<size_t>(n_chunks), 0);
  uint64_t total = 0, total_bytes = 0;
  bool reseed = false;
  // grows a buffer that outlives the per-chunk handles and their streams (plain allocation), keeping `used` bytes
  auto grow = [](DevBuf* b, size_t need, size_t used) -> int {
    if (need <= b->bytes) return PA_OK;
    DevBuf bigger;
    bigger.plain = true;
    PA_TRY(bigger.alloc(std::max<size_t>(need * 2, 1u << 20), nullptr));
    if (used) CUDA_TRY(cudaMemcpy(bigger.p, b->p, used, cudaMemcpyDeviceToDevice));
    *b = std::move(bigger);
    return PA_OK;
  };
  for (int64_t c = 0; c < n_chunks && !reseed; ++c) {
    const int64_t lo = c * chunk_rows, len = std::min(chunk_rows, n - lo);
    std::vector<ArrowDeviceArray> kc(keys, keys + n_keys);   // views: same buffers, shifted window
    ArrowDeviceArray vc = *values;
    for (ArrowDeviceArray& k : kc) {
      k.array.offset += lo; k.array.length = len;
      if (k.array.null_count > 0) k.array.null_count = -1;
      k.array.release = nullptr;
    }
    vc.array.offset += lo; vc.array.length = len;
    if (vc.array.null_count > 0) vc.array.null_count = -1;
    vc.array.release = nullptr;
    o.row_base = base0 + lo;
    pa_groupby* h = nullptr;
    PA_TRY(pa_groupby_create(kc.data(), key_schemas, n_keys, &o, &h));
    HandlePtr guard(h);
    if (composite) {
      pa_key_layout mine;
      fields_layout(h, &mine);
      for (int j = 0; j < n_keys; ++j)
        if (mine.width[j] != whole.width[j] || mine.bits[j] != whole.bits[j] || mine.nullable[j] != whole.nullable[j])
          return set_err(PA_ERR_STATE, "chunk %lld packs key column %d differently from the whole column", (long long)c, j);
    }
    if (str) PA_TRY(set_key_seed(h, seed));
    PA_TRY(pa_groupby_aggregate(h, &vc, value_schema, agg_mask));
    if (str && h->key_seed != seed) {   // this chunk's own check moved the seed
      seed = h->key_seed;
      reseed = true;
      break;
    }
    int64_t cnt = 0, nbytes = 0;
    if (str) PA_TRY(pa_groupby_partials_count_utf8(h, 1, &cnt, &nbytes));
    else PA_TRY(pa_groupby_partials_count(h, 1, &cnt));
    counts[static_cast<size_t>(c)] = cnt;
    PA_TRY(grow(&records, (total + static_cast<uint64_t>(cnt)) * RW * 8, total * RW * 8));
    if (str) {
      PA_TRY(grow(&lengths, (total + static_cast<uint64_t>(cnt)) * 4, total * 4));
      PA_TRY(grow(&bytes, total_bytes + static_cast<uint64_t>(nbytes), total_bytes));
    }
    if (cnt) {
      uint64_t* recs = reinterpret_cast<uint64_t*>(static_cast<char*>(records.p) + total * RW * 8);
      PA_TRY(partials_export(h, 1, recs, cnt, RW));
      if (str) {
        DevBuf off, tmp;
        PA_TRY(keystr_export(h, recs, RW, static_cast<uint64_t>(cnt), lengths.as<uint32_t>() + total, bytes.as<uint8_t>() + total_bytes, &off, &tmp));
      }
    }
    PA_TRY(pa_groupby_sync(h));
    total += static_cast<uint64_t>(cnt);
    total_bytes += static_cast<uint64_t>(nbytes);
  }
  if (reseed) continue;
  o.row_base = base0;
  const std::string kfmt = composite ? "L" : key_schemas->format;
  pa_groupby* m = nullptr;
  PA_TRY(pa_merge_create(records.p, counts.data(), static_cast<int32_t>(n_chunks), agg_mask, value_schema->format, kfmt.c_str(), &o, &m));
  HandlePtr merged(m);
  if (composite) {
    std::vector<const char*> kf;
    for (int j = 0; j < n_keys; ++j) kf.push_back(key_schemas[j].format);
    PA_TRY(set_merged_layout(m, whole, kf.data()));
  }
  if (str) {
    bool collided = false;
    PA_TRY(merge_key_strings(m, records.as<uint64_t>(), RW, total, lengths.as<uint32_t>(), bytes.as<uint8_t>(), total_bytes, &collided));
    if (collided) {
      ++seed;
      continue;
    }
  }
  CUDA_TRY(cudaDeviceSynchronize());   // `records` is released on return
  *merged_out = merged.release();
  return PA_OK;
  }
}

// ---- multi-GPU through the C ABI: communicator + the whole sharded step (SURVEY.md §8b "multi-GPU variants taking a
// communicator handle", §8e) ----
struct pa_comm {
  ncclComm_t comm = nullptr;
  int world = 1, rank = 0, device = 0;
  bool own = false;
  DevBuf send, recv, d_counts, d_all, d_cursor;     // kept between steps (grow only)
  DevBuf psend, precv, pset;                        // count_distinct: distinct pairs sent / received, the owner's set
  MergeScratch merge;
  DevBuf layouts;                                   // composite keys: this rank's pa_key_layout, then all ranks'
  double phase_ms[5] = {0, 0, 0, 0, 0};   // last step: local pass, count + export, exchange, merge, total
  double agree_ms = 0, repack_ms = 0;     // last step: key layout gather, repack (pa_comm_last_key_layout)
  cudaEvent_t ev[8] = {};
  uint64_t h_bound = 0;                   // end of this rank's row shard (staging for the async copy)
  int last_record_bytes = 0, last_unordered = 0;   // pa_comm_last_exchange
  int64_t last_table_slots = 0;
  int64_t last_pairs_sent = 0, last_pairs_received = 0, last_set_slots = 0;   // pa_comm_last_distinct
  // utf8 key: lengths and key bytes sent / received, scratch of the byte offsets, the collision word of the all-reduce
  DevBuf ksend_len, krecv_len, ksend_bytes, krecv_bytes, koff, ktmp, kflag;
  uint64_t h_seed = 0;                    // (staging for the async copies)
  uint32_t h_flag = 0;
  int64_t last_bytes_sent = 0, last_bytes_received = 0;   // pa_comm_last_key_strings
  uint64_t last_seed = 0;
  int32_t last_attempts = 0;
};

#define NCCL_TRY(expr)                                                                                          \
  do {                                                                                                          \
    ncclResult_t r__ = (expr);                                                                                  \
    if (r__ != ncclSuccess) return set_err(PA_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, ncclGetErrorString(r__), __FILE__, __LINE__); \
  } while (0)

int pa_comm_unique_id(void* out_id, int64_t capacity_bytes) {
  if (!out_id || capacity_bytes < static_cast<int64_t>(sizeof(ncclUniqueId))) return set_err(PA_ERR_INVALID, "id buffer must hold %zu bytes", sizeof(ncclUniqueId));
  ncclUniqueId id;
  NCCL_TRY(ncclGetUniqueId(&id));
  memcpy(out_id, &id, sizeof id);
  return PA_OK;
}

static int comm_finish(pa_comm* c) {
  // The communicator outlives the handles (and their streams) it is used with: its scratch does not belong to any
  // stream's allocation order.
  for (DevBuf* b : {&c->send, &c->recv, &c->d_counts, &c->d_all, &c->d_cursor, &c->psend, &c->precv, &c->pset, &c->layouts, &c->merge.tkeys, &c->merge.idx,
                    &c->merge.m_first, &c->merge.m_slot, &c->merge.s_first, &c->merge.s_slot, &c->merge.cub_tmp, &c->ksend_len, &c->krecv_len,
                    &c->ksend_bytes, &c->krecv_bytes, &c->koff, &c->ktmp, &c->kflag})
    b->plain = true;
  for (auto& e : c->ev) CUDA_TRY(cudaEventCreate(&e));
  return PA_OK;
}

int pa_comm_create(const void* id, int32_t world, int32_t rank, int32_t device, pa_comm** out) {
  if (!id || !out || world < 1 || world > 64 || rank < 0 || rank >= world) return set_err(PA_ERR_INVALID, "pa_comm_create: bad argument (1 <= world <= 64)");
  std::unique_ptr<pa_comm> c(new pa_comm());
  c->world = world; c->rank = rank; c->device = device; c->own = true;
  CUDA_TRY(cudaSetDevice(device));
  ncclUniqueId uid;
  memcpy(&uid, id, sizeof uid);
  NCCL_TRY(ncclCommInitRank(&c->comm, world, uid, rank));
  PA_TRY(comm_finish(c.get()));
  *out = c.release();
  return PA_OK;
}

int pa_comm_adopt(void* nccl_comm, int32_t world, int32_t rank, int32_t device, pa_comm** out) {
  if (!nccl_comm || !out || world < 1 || world > 64 || rank < 0 || rank >= world) return set_err(PA_ERR_INVALID, "pa_comm_adopt: bad argument");
  std::unique_ptr<pa_comm> c(new pa_comm());
  c->comm = static_cast<ncclComm_t>(nccl_comm);
  c->world = world; c->rank = rank; c->device = device; c->own = false;
  CUDA_TRY(cudaSetDevice(device));
  PA_TRY(comm_finish(c.get()));
  *out = c.release();
  return PA_OK;
}

void pa_comm_destroy(pa_comm* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (auto& e : c->ev) if (e) cudaEventDestroy(e);
  if (c->own && c->comm) ncclCommDestroy(c->comm);
  delete c;
}

int pa_comm_last_exchange(pa_comm* c, int32_t* record_bytes, int32_t* unordered_export, int64_t* merge_table_slots) {
  if (!c) return set_err(PA_ERR_INVALID, "null argument");
  if (record_bytes) *record_bytes = c->last_record_bytes;
  if (unordered_export) *unordered_export = c->last_unordered;
  if (merge_table_slots) *merge_table_slots = c->last_table_slots;
  return PA_OK;
}

int pa_comm_last_distinct(pa_comm* c, int64_t* pairs_sent, int64_t* pairs_received, int64_t* set_slots) {
  if (!c) return set_err(PA_ERR_INVALID, "null argument");
  if (pairs_sent) *pairs_sent = c->last_pairs_sent;
  if (pairs_received) *pairs_received = c->last_pairs_received;
  if (set_slots) *set_slots = c->last_set_slots;
  return PA_OK;
}

int pa_comm_last_key_layout(pa_comm* c, double* agree_ms, double* repack_ms) {
  if (!c) return set_err(PA_ERR_INVALID, "null argument");
  if (agree_ms) *agree_ms = c->agree_ms;
  if (repack_ms) *repack_ms = c->repack_ms;
  return PA_OK;
}

int pa_comm_last_key_strings(pa_comm* c, int64_t* bytes_sent, int64_t* bytes_received, uint64_t* seed, int32_t* attempts) {
  if (!c) return set_err(PA_ERR_INVALID, "null argument");
  if (bytes_sent) *bytes_sent = c->last_bytes_sent;
  if (bytes_received) *bytes_received = c->last_bytes_received;
  if (seed) *seed = c->last_seed;
  if (attempts) *attempts = c->last_attempts;
  return PA_OK;
}

int pa_comm_last_phases(pa_comm* c, double phase_ms[5]) {
  if (!c || !phase_ms) return set_err(PA_ERR_INVALID, "null argument");
  for (int i = 0; i < 5; ++i) phase_ms[i] = c->phase_ms[i];
  return PA_OK;
}

// Grouped send / receive of `words`-word records: send_cnt[p] from `send` (grouped by destination) to every rank p,
// recv_cnt[p] from rank p into `recv` (grouped by source).  Every rank issues the same calls in the same order.
static int exchange_grouped(pa_comm* c, cudaStream_t st, const uint64_t* send, const int64_t* send_cnt, uint64_t* recv,
                            const int64_t* recv_cnt, size_t words) {
  NCCL_TRY(ncclGroupStart());
  uint64_t so = 0, ro = 0;
  for (int p = 0; p < c->world; ++p) {
    if (send_cnt[p]) NCCL_TRY(ncclSend(send + so * words, static_cast<size_t>(send_cnt[p]) * words, ncclUint64, p, c->comm, st));
    if (recv_cnt[p]) NCCL_TRY(ncclRecv(recv + ro * words, static_cast<size_t>(recv_cnt[p]) * words, ncclUint64, p, c->comm, st));
    so += send_cnt[p];
    ro += recv_cnt[p];
  }
  NCCL_TRY(ncclGroupEnd());
  return PA_OK;
}

// One multi-GPU step for this rank: local stages 1-3 on its row shard -> partial records bucketed by owner =
// hash(key) % world -> counts (ncclAllGather) and records (grouped ncclSend / ncclRecv: NCCL 2.27 has no all-to-all
// primitive) over NVLink -> owner-side merge in source-rank order.  Everything runs on the handle's stream.
int pa_groupby_sharded_aggregate(pa_groupby* g, pa_comm* c, const struct ArrowDeviceArray* values,
                                 const struct ArrowSchema* value_schema, uint32_t agg_mask, pa_groupby** merged_out) {
  if (!g || !c || !values || !value_schema || !merged_out) return set_err(PA_ERR_INVALID, "null argument");
  if (agg_mask == 0 || (agg_mask & ~SHARDED_AGGS))
    return set_err(PA_ERR_NOT_IMPLEMENTED, "sharded aggregates: sum / mean / count / min / max / first / last / product / variance / stddev / "
                                           "all / any / count_distinct");
  if (g->device != c->device) return set_err(PA_ERR_INVALID, "handle lives on device %d, communicator on %d", g->device, c->device);
  PA_TRY(ensure_device(g));
  cudaStream_t st = g->stream;
  const int W = c->world;
  // 0. composite key: every rank's key layout to everybody, one agreed layout, repack when it differs from this
  // handle's.  On every step (never cached): a rank that skipped the gather while another ran it would hang the step.
  // A rank that cannot describe its layout still takes part (with n_keys = 0), so that every rank fails together.  That
  // includes a rank whose composite key is hashed (whether a key packs depends on the shard's own nulls and
  // dictionaries), so the branch is taken on the number of key columns.
  const bool composite = !g->resample && g->keys.size() > 1;
  pa_key_layout agreed{};
  c->agree_ms = 0; c->repack_ms = 0;
  if (composite) {
    pa_key_layout mine{};
    const int mine_rc = key_layout_of(g, &mine);
    const std::string mine_err = mine_rc != PA_OK ? g_err : std::string();
    if (mine_rc != PA_OK) mine = pa_key_layout{};
    const size_t LB = sizeof(pa_key_layout);
    PA_TRY(c->layouts.alloc(LB * (W + 1), st));
    CUDA_TRY(cudaEventRecord(c->ev[5], st));
    CUDA_TRY(cudaMemcpyAsync(c->layouts.p, &mine, LB, cudaMemcpyHostToDevice, st));
    NCCL_TRY(ncclAllGather(c->layouts.p, c->layouts.as<char>() + LB, LB, ncclUint8, c->comm, st));
    std::vector<pa_key_layout> all(static_cast<size_t>(W));
    CUDA_TRY(cudaMemcpyAsync(all.data(), c->layouts.as<char>() + LB, LB * W, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaEventRecord(c->ev[6], st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (mine_rc != PA_OK) return set_err(mine_rc, "%s", mine_err.c_str());
    PA_TRY(pa_key_layout_agree(all.data(), W, &agreed));
    bool repack = false;
    for (int j = 0; j < agreed.n_keys; ++j) repack = repack || agreed.nullable[j] != mine.nullable[j];
    PA_TRY(pa_groupby_set_key_layout(g, &agreed));
    float t = 0;
    CUDA_TRY(cudaEventElapsedTime(&t, c->ev[5], c->ev[6]));
    c->agree_ms = t;
    if (repack) {
      CUDA_TRY(cudaEventRecord(c->ev[7], st));
      CUDA_TRY(cudaEventSynchronize(c->ev[7]));
      CUDA_TRY(cudaEventElapsedTime(&t, c->ev[6], c->ev[7]));
      c->repack_ms = t;
    }
  }
  // utf8 key: the records carry the hash of the key bytes, and the bytes travel with them (strkeys.cuh).  Every rank
  // must hash with the same seed, and no owner may see two strings under one hash: the count gather carries every
  // rank's seed, and after the owner's byte check one all-reduce tells every rank whether some owner saw a collision.
  // Either way all ranks redo the step together with the agreed (max) or the next seed, four seeds at most; every such
  // branch is taken on gathered values only.
  const bool str = is_str_key(g);
  c->last_bytes_sent = 0; c->last_bytes_received = 0; c->last_attempts = 0;
  for (int attempt = 1;; ++attempt) {
  CUDA_TRY(cudaEventRecord(c->ev[0], st));
  // 1. local pass.  sum / mean of floats / count need one 32-byte sector per group (compact records, merge.cuh),
  // everything else the full record; with compact records the bucketed path may hand over its unordered group records
  // as they are (the merge orders by global first row anyway).  Product / variance / stddev: the local pass runs its
  // second stage too, and the records carry its terms (REC_WORDS_STAGE2).  All / any travel in the full record's
  // min / max words.  Count_distinct: the local pass keeps its distinct pairs, which take a second exchange to their
  // owners (pairs are counted per owner with the records, exported in [1], sent in [2], deduplicated in [3]).
  int vw_ = 8, vc_ = VC_I;
  PA_TRY(parse_format(value_schema->format, &vw_, &vc_));
  const bool stage2 = (agg_mask & PA_AGG_STAGE2) != 0;
  const bool distinct = (agg_mask & PA_AGG_COUNT_DISTINCT) != 0;
  const bool full_only = stage2 || distinct || (agg_mask & (PA_AGG_BOOL_ALL | PA_AGG_BOOL_ANY));
  const bool compact = !full_only && !is_wide(agg_mask, vc_) && !(agg_mask & (AGG_FIRST | AGG_LAST));
  // (a utf8 key's first pass checks its grouping byte for byte, which reads the ordered groups)
  g->want_unordered = compact && !g->resample && (!str || g->key_verified);
  const int local_rc = aggregate_entry(g, values, value_schema, agg_mask, false);
  g->want_unordered = false;
  if (local_rc != PA_OK) return local_rc;
  const bool unordered = g->unordered;
  g->unordered = false;
  const uint32_t G_local = unordered ? g->unordered_G : g->G;
  if (unordered && g->opt.expected_groups <= 0) g->opt.expected_groups = std::max<int64_t>(G_local, 1);   // (the keys of a handle never change)
  CUDA_TRY(cudaEventRecord(c->ev[1], st));
  // 2. counts per owner, all ranks' counts to everybody
  // (every rank also tells the others where its row shard ends: the merge orders by GLOBAL first row and only has
  // to sort the bits below the largest one)
  // (count_distinct: the W pair counts per owner follow, at [W + 1, 2 W + 1), in the same gather)
  // (utf8 key: then the rank's hash seed and its W key byte counts per owner, at KS and [KS + 1, KS + 1 + W))
  const int KS = W + 1 + (distinct ? W : 0);
  const int W1 = KS + (str ? 1 + W : 0);
  PA_TRY(c->d_counts.alloc(sizeof(uint64_t) * W1, st));
  PA_TRY(c->d_all.alloc(sizeof(uint64_t) * W1 * W, st));
  CUDA_TRY(cudaMemsetAsync(c->d_counts.p, 0, sizeof(uint64_t) * W1, st));
  c->h_bound = static_cast<uint64_t>(g->opt.row_base) + static_cast<uint64_t>(g->n);
  CUDA_TRY(cudaMemcpyAsync(c->d_counts.as<uint64_t>() + W, &c->h_bound, sizeof(uint64_t), cudaMemcpyHostToDevice, st));
  if (unordered) {
    if (G_local) {
      k_bkrec_count<<<(G_local + 255) / 256, 256, 0, st>>>(static_cast<const BkRec32*>(g->unordered_recs), G_local, static_cast<uint32_t>(W), c->d_counts.as<unsigned long long>());
      CUDA_TRY(cudaGetLastError());
    }
  } else {
    PA_TRY(partials_count_async(g, W, c->d_counts.as<unsigned long long>()));
  }
  if (distinct) PA_TRY(pairs_count_async(g, W, c->d_counts.as<unsigned long long>() + W + 1));
  if (str) {
    c->h_seed = g->key_seed;
    CUDA_TRY(cudaMemcpyAsync(c->d_counts.as<uint64_t>() + KS, &c->h_seed, sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    PA_TRY(keystr_count_async(g, W, unordered ? g->unordered_recs : nullptr, G_local, c->d_counts.as<unsigned long long>() + KS + 1));
  }
  NCCL_TRY(ncclAllGather(c->d_counts.p, c->d_all.p, W1, ncclUint64, c->comm, st));
  std::vector<uint64_t> all(static_cast<size_t>(W1) * W);
  CUDA_TRY(cudaMemcpyAsync(all.data(), c->d_all.p, sizeof(uint64_t) * W1 * W, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  if (str) {   // a rank whose own check moved its seed: everybody takes the largest seed and redoes the step
    uint64_t lo = ~0ull, hi = 0;
    for (int p = 0; p < W; ++p) {
      lo = std::min(lo, all[static_cast<size_t>(p) * W1 + KS]);
      hi = std::max(hi, all[static_cast<size_t>(p) * W1 + KS]);
    }
    if (hi >= 4) return set_err(PA_ERR_STATE, "utf8 keys: four differently seeded 64-bit hashes all collided");
    if (lo != hi) {
      PA_TRY(set_key_seed(g, hi));
      continue;
    }
  }
  std::vector<int64_t> send_cnt(W), recv_cnt(W), psend_cnt(W, 0), precv_cnt(W, 0), ksend_cnt(W, 0), krecv_cnt(W, 0);
  uint64_t send_total = 0, recv_total = 0, row_bound = 1, psend_total = 0, precv_total = 0, ksend_total = 0, krecv_total = 0;
  for (int p = 0; p < W; ++p) {
    send_cnt[p] = static_cast<int64_t>(all[static_cast<size_t>(c->rank) * W1 + p]);
    recv_cnt[p] = static_cast<int64_t>(all[static_cast<size_t>(p) * W1 + c->rank]);
    send_total += send_cnt[p];
    recv_total += recv_cnt[p];
    row_bound = std::max(row_bound, all[static_cast<size_t>(p) * W1 + W]);
    if (distinct) {
      psend_cnt[p] = static_cast<int64_t>(all[static_cast<size_t>(c->rank) * W1 + W + 1 + p]);
      precv_cnt[p] = static_cast<int64_t>(all[static_cast<size_t>(p) * W1 + W + 1 + c->rank]);
      psend_total += psend_cnt[p];
      precv_total += precv_cnt[p];
    }
    if (str) {
      ksend_cnt[p] = static_cast<int64_t>(all[static_cast<size_t>(c->rank) * W1 + KS + 1 + p]);
      krecv_cnt[p] = static_cast<int64_t>(all[static_cast<size_t>(p) * W1 + KS + 1 + c->rank]);
      ksend_total += ksend_cnt[p];
      krecv_total += krecv_cnt[p];
    }
  }
  // (checked for every owner: every rank sees every count, so all ranks fail together before any record is sent)
  for (int q = 0; distinct && q < W; ++q) {
    uint64_t to_q = 0;
    for (int p = 0; p < W; ++p) to_q += all[static_cast<size_t>(p) * W1 + W + 1 + q];
    if (to_q > 0xFFFFFFFEull) return set_err(PA_ERR_INVALID, "rank %d would receive more than 2^32 - 2 distinct pairs in one merge", q);
  }
  // 3. export the records grouped by owner
  const int words = record_words(agg_mask, compact);
  const size_t RW = static_cast<size_t>(words);
  PA_TRY(c->send.alloc(std::max<uint64_t>(send_total, 1) * RW * 8, st));
  PA_TRY(c->recv.alloc(std::max<uint64_t>(recv_total, 1) * RW * 8, st));
  if (unordered) {
    PA_TRY(owner_cursors(st, send_cnt.data(), W, &c->d_cursor));
    if (G_local) {
      k_bkrec_scatter<<<(G_local + 255) / 256, 256, 0, st>>>(static_cast<const BkRec32*>(g->unordered_recs), G_local, static_cast<uint32_t>(W),
                                                             g->opt.row_base, c->d_cursor.as<unsigned long long>(), c->send.as<uint64_t>());
      CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaStreamSynchronize(st));
  } else {
    g->parts_n = W;
    g->parts_counts.assign(send_cnt.begin(), send_cnt.end());
    PA_TRY(partials_export(g, W, c->send.p, static_cast<int64_t>(std::max<uint64_t>(send_total, g->G)), words));
  }
  const size_t PW = DP_WORDS;
  if (distinct) {
    PA_TRY(c->psend.alloc(std::max<uint64_t>(psend_total, 1) * PW * 8, st));
    PA_TRY(c->precv.alloc(std::max<uint64_t>(precv_total, 1) * PW * 8, st));
    PA_TRY(pairs_export(g, W, psend_cnt.data(), c->psend.p, &c->d_cursor));
  }
  if (str) {   // lengths and key bytes of the records just written, in the same owner segments
    PA_TRY(c->ksend_len.alloc(std::max<uint64_t>(send_total, 1) * 4, st));
    PA_TRY(c->krecv_len.alloc(std::max<uint64_t>(recv_total, 1) * 4, st));
    PA_TRY(c->ksend_bytes.alloc(std::max<uint64_t>(ksend_total, 1), st));
    PA_TRY(c->krecv_bytes.alloc(std::max<uint64_t>(krecv_total, 1), st));
    PA_TRY(keystr_export(g, c->send.as<uint64_t>(), words, send_total, c->ksend_len.as<uint32_t>(), c->ksend_bytes.as<uint8_t>(), &c->koff, &c->ktmp));
  }
  CUDA_TRY(cudaEventRecord(c->ev[2], st));
  // 4. all-to-all of the records; the distinct pairs, grouped by owner, in a second exchange; a utf8 key's lengths and
  // bytes in one more
  PA_TRY(exchange_grouped(c, st, c->send.as<uint64_t>(), send_cnt.data(), c->recv.as<uint64_t>(), recv_cnt.data(), RW));
  if (distinct) PA_TRY(exchange_grouped(c, st, c->psend.as<uint64_t>(), psend_cnt.data(), c->precv.as<uint64_t>(), precv_cnt.data(), PW));
  if (str) {
    NCCL_TRY(ncclGroupStart());
    uint64_t so = 0, ro = 0, sb = 0, rb = 0;
    for (int p = 0; p < W; ++p) {
      if (send_cnt[p]) NCCL_TRY(ncclSend(c->ksend_len.as<uint32_t>() + so, static_cast<size_t>(send_cnt[p]), ncclUint32, p, c->comm, st));
      if (recv_cnt[p]) NCCL_TRY(ncclRecv(c->krecv_len.as<uint32_t>() + ro, static_cast<size_t>(recv_cnt[p]), ncclUint32, p, c->comm, st));
      if (ksend_cnt[p]) NCCL_TRY(ncclSend(c->ksend_bytes.as<uint8_t>() + sb, static_cast<size_t>(ksend_cnt[p]), ncclUint8, p, c->comm, st));
      if (krecv_cnt[p]) NCCL_TRY(ncclRecv(c->krecv_bytes.as<uint8_t>() + rb, static_cast<size_t>(krecv_cnt[p]), ncclUint8, p, c->comm, st));
      so += send_cnt[p]; ro += recv_cnt[p]; sb += ksend_cnt[p]; rb += krecv_cnt[p];
    }
    NCCL_TRY(ncclGroupEnd());
  }
  CUDA_TRY(cudaEventRecord(c->ev[3], st));
  // 5. owner-side merge
  const std::string kfmt = g->resample ? g->index_format : composite ? "L" : g->keys[0].format;
  HandlePtr m(new pa_groupby());
  pa_options mo;
  pa_options_init(&mo);
  mo.device = g->device;
  mo.cuda_stream = st;
  PA_TRY(handle_init(m.get(), &mo));
  PA_TRY(merge_counted(m.get(), c->recv.p, recv_cnt.data(), W, agg_mask & ~PA_AGG_COUNT_DISTINCT, value_schema->format, kfmt.c_str(),
                       &c->merge, row_bound, compact));
  if (composite) {
    std::vector<const char*> kf;
    for (const Column& k : g->keys) kf.push_back(k.format.c_str());
    PA_TRY(set_merged_layout(m.get(), agreed, kf.data()));
  }
  if (str) {   // the owner's byte check, then every rank learns whether any owner saw two strings under one hash
    bool collided = false;
    PA_TRY(merge_key_strings(m.get(), c->recv.as<uint64_t>(), words, recv_total, c->krecv_len.as<uint32_t>(), c->krecv_bytes.as<uint8_t>(),
                             krecv_total, &collided));
    c->h_flag = collided ? 1u : 0u;
    PA_TRY(c->kflag.alloc(4, st));
    CUDA_TRY(cudaMemcpyAsync(c->kflag.p, &c->h_flag, 4, cudaMemcpyHostToDevice, st));
    NCCL_TRY(ncclAllReduce(c->kflag.p, c->kflag.p, 1, ncclUint32, ncclMax, c->comm, st));
    CUDA_TRY(cudaMemcpyAsync(&c->h_flag, c->kflag.p, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    c->last_bytes_sent = static_cast<int64_t>(ksend_total);
    c->last_bytes_received = static_cast<int64_t>(krecv_total);
    c->last_seed = g->key_seed;
    c->last_attempts = attempt;
    if (c->h_flag) {
      if (g->key_seed + 1 >= 4) return set_err(PA_ERR_STATE, "utf8 keys: four differently seeded 64-bit hashes all collided");
      PA_TRY(set_key_seed(g, g->key_seed + 1));
      continue;
    }
  }
  uint64_t set_slots = 0;
  if (distinct) PA_TRY(merge_distinct(m.get(), c->precv.p, precv_total, &c->pset, &set_slots));
  CUDA_TRY(cudaEventRecord(c->ev[4], st));
  CUDA_TRY(cudaEventSynchronize(c->ev[4]));
  float t = 0;
  for (int i = 0; i < 4; ++i) { CUDA_TRY(cudaEventElapsedTime(&t, c->ev[i], c->ev[i + 1])); c->phase_ms[i] = t; }
  CUDA_TRY(cudaEventElapsedTime(&t, c->ev[0], c->ev[4]));
  c->phase_ms[4] = t;
  c->last_record_bytes = static_cast<int>(RW * 8);
  c->last_unordered = unordered ? 1 : 0;
  c->last_table_slots = static_cast<int64_t>(c->merge.last_slots);
  c->last_pairs_sent = static_cast<int64_t>(psend_total);
  c->last_pairs_received = static_cast<int64_t>(precv_total);
  c->last_set_slots = static_cast<int64_t>(set_slots);
  *merged_out = m.release();
  return PA_OK;
  }
}

// ---- synthetic generator ----
static int synth_grid(int64_t n) {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return static_cast<int>(std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, static_cast<int64_t>(sms) * 16)));
}
int pa_synth_keys_i64(void* dev_out, int64_t n, int64_t first_row, uint64_t n_groups, uint64_t seed, void* cuda_stream) {
  if (!dev_out || n_groups == 0) return set_err(PA_ERR_INVALID, "bad argument");
  k_synth_keys<<<synth_grid(n), 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(static_cast<int64_t*>(dev_out), n, first_row, n_groups, seed);
  CUDA_TRY(cudaGetLastError());
  return PA_OK;
}
int pa_synth_vals_f64(void* dev_out, int64_t n, int64_t first_row, uint64_t seed, void* cuda_stream) {
  if (!dev_out) return set_err(PA_ERR_INVALID, "bad argument");
  k_synth_vals<<<synth_grid(n), 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(static_cast<double*>(dev_out), n, first_row, seed);
  CUDA_TRY(cudaGetLastError());
  return PA_OK;
}
int pa_synth_validity(void* dev_bitmap_out, int64_t n, int64_t first_row, uint64_t seed, uint32_t null_every, void* cuda_stream) {
  if (!dev_bitmap_out || null_every == 0) return set_err(PA_ERR_INVALID, "bad argument");
  k_synth_validity<<<synth_grid((n + 7) / 8), 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(static_cast<uint8_t*>(dev_bitmap_out), n, first_row, seed, null_every);
  CUDA_TRY(cudaGetLastError());
  return PA_OK;
}
int pa_synth_timestamps(void* dev_out, int64_t n, int64_t first_row, int64_t t0_ns, int64_t step_ns, uint64_t seed, void* cuda_stream) {
  if (!dev_out || step_ns <= 0) return set_err(PA_ERR_INVALID, "bad argument");
  k_synth_ts<<<synth_grid(n), 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(static_cast<int64_t*>(dev_out), n, first_row, t0_ns, step_ns, seed);
  CUDA_TRY(cudaGetLastError());
  return PA_OK;
}

}  // extern "C"
