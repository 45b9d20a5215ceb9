// Device-side result of stages 1-3: one entry per group, first-appearance order.
#pragma once
#include "common.cuh"

namespace pa {

// key_kind values
constexpr uint8_t KK_REGULAR = 0;   // key[] holds the packed 64-bit key
constexpr uint8_t KK_NULL = 1;      // the null-key group (single-key mode)

struct GroupResult {
  uint64_t* key;        // packed key
  uint8_t* key_kind;    // KK_*
  uint64_t* sum;        // raw bits: double (VC_F) or wrapping (u)int64
  double* dsum;         // sum of values converted to double (VC_I / VC_U mean); may be null for VC_F
  uint32_t* count;      // non-null values
  uint64_t* count64;    // merged (multi-GPU) results only: 64-bit counts, overrides `count` when non-null
  uint32_t* first_row;  // local row index of the first / last row of the group
  uint32_t* last_row;
  uint64_t* min_ord;    // order-mapped min / max over non-null, non-NaN values
  uint64_t* max_ord;
};

// status words shared by the scan / merge kernels and read back by the host
constexpr int ST_OVERFLOW = 0;   // table capacity exceeded -> caller retries on a bigger path
constexpr int ST_NGROUPS = 1;
constexpr int ST_UNSORTED = 2;   // resample: timestamps not sorted
constexpr int ST_COUNTER = 3;    // scratch append counter
constexpr int ST_DENSE_MISS = 4; // low-cardinality dense mode met a key outside its window -> rerun in hash mode
constexpr int ST_PEER_OVERFLOW = 4;  // merge of padded blocks: a source had more groups than a block holds (own status buffer)
constexpr int ST_NO_TERMS = 2;    // merge of stage-2 records: a record lacks the variance / product terms asked for (own status buffer)
constexpr int ST_ABORT = 5;      // some CTA gave up (overflow / dense miss): the others stop early, merge is skipped
constexpr int ST_MODE = 6;       // low-cardinality scan: 1 dense, 2 hash
constexpr int ST_RLOG = 7;       // low-cardinality scan: log2 of the accumulator replication
constexpr int ST_WORDS = 8;

// Range of a sample of the key column (signed order), accumulated with atomicMax by any grid:
//   nmin_ord = max over sampled valid keys of ~ord(key), max_ord = max of ord(key), ord = key ^ 2^63.
// Zero-initialised by the host; both zero = no valid key sampled.
struct KeyRange {
  unsigned long long nmin_ord;
  unsigned long long max_ord;
};

// Called by every thread of a grid of `nt` threads (thread index t): samples row floor(t * n / nt).
__device__ __forceinline__ void key_range_sample(const void* keys, const uint8_t* kvalid, int64_t koff, int kw, int64_t n,
                                                 uint32_t t, uint32_t nt, KeyRange* out) {
  uint64_t nmin = 0, mx = 0;
  const int64_t r = n <= static_cast<int64_t>(nt) ? static_cast<int64_t>(t)
                                                 : static_cast<int64_t>((static_cast<uint64_t>(t) * static_cast<uint64_t>(n)) / nt);
  if (r < n && (!kvalid || bit_at(kvalid, koff + r))) {
    const uint64_t key = kw == 8 ? static_cast<const uint64_t*>(keys)[r]
                                 : static_cast<uint64_t>(static_cast<const uint32_t*>(keys)[r]);
    const uint64_t o = key ^ 0x8000000000000000ull;
    nmin = ~o;
    mx = o;
  }
#pragma unroll
  for (int d = 16; d; d >>= 1) {
    const uint64_t on = __shfl_xor_sync(0xFFFFFFFFu, nmin, d), om = __shfl_xor_sync(0xFFFFFFFFu, mx, d);
    nmin = on > nmin ? on : nmin;
    mx = om > mx ? om : mx;
  }
  if (lane_id() == 0 && (nmin | mx)) {
    atomicMax(&out->nmin_ord, static_cast<unsigned long long>(nmin));
    atomicMax(&out->max_ord, static_cast<unsigned long long>(mx));
  }
}

// Decodes a KeyRange: false when nothing was sampled; else the smallest sampled key and the span (max - min).
__device__ __forceinline__ bool key_range_get(const KeyRange* p, uint64_t* smin, uint64_t* span) {
  const uint64_t a = p->nmin_ord, b = p->max_ord;
  if (a == 0 && b == 0) return false;
  *smin = (~a) ^ 0x8000000000000000ull;
  *span = (b ^ 0x8000000000000000ull) - *smin;   // max >= min in signed order, so this does not wrap
  return true;
}

}  // namespace pa
