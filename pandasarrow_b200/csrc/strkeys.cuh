// utf8 / large_utf8 key columns on the device (SURVEY.md §8b: buffers[1] = offsets, buffers[2] = bytes).
// makeGroups groups any key type through arrow's Grouper (/root/reference/src/dataframe.cpp:1579-1584) and the
// reference's golden tests key on strings (tests/cudf_examples/dataframe_resample_test.cpp:8-69); round 1
// dictionary-encoded such keys on the HOST.  Here:
//   k_str_hash    every row's string -> a seeded 64-bit hash; the ordinary stages 1-3 then run on that 8-byte column
//   exactness: every row's bytes are compared with the bytes of its group's first row (the group's representative,
//              k_row_verify in rowkeys.cuh); two different strings with one hash set a flag and the host re-hashes the
//              column with another seed (probability ~ n_groups^2 / 2^65 per attempt)
//   k_str_lengths / k_str_gather   unique(): lengths of the representatives -> offsets (scan) -> bytes
#pragma once
#include "bucketed.cuh"
#include "rowids.cuh"

namespace pa {

struct StrCol {
  const void* offsets;       // int32 or int64, already advanced by the array offset
  const uint8_t* bytes;
  int wide;                  // 1 = int64 offsets (large_utf8)
};

__device__ __forceinline__ int64_t str_off(const StrCol& c, int64_t i) {
  return c.wide ? static_cast<const int64_t*>(c.offsets)[i] : static_cast<int64_t>(static_cast<const int32_t*>(c.offsets)[i]);
}

// 64-bit hash of a byte string: 8 bytes per step through a multiply-xorshift mix (wyhash-like), length folded in.
__device__ __forceinline__ uint64_t str_hash64(const uint8_t* p, int64_t len, uint64_t seed) {
  uint64_t h = seed ^ (static_cast<uint64_t>(len) * 0x9E3779B97F4A7C15ull);
  int64_t i = 0;
  for (; i + 8 <= len; i += 8) {
    uint64_t w = 0;
#pragma unroll
    for (int b = 0; b < 8; ++b) w |= static_cast<uint64_t>(p[i + b]) << (8 * b);
    h = (h ^ w) * 0xFF51AFD7ED558CCDull;
    h ^= h >> 32;
  }
  uint64_t w = 0;
  for (int b = 0; i < len; ++i, ++b) w |= static_cast<uint64_t>(p[i]) << (8 * b);
  h = (h ^ w) * 0xC4CEB9FE1A85EC53ull;
  h ^= h >> 29;
  h *= 0x94D049BB133111EBull;
  return h ^ (h >> 32);
}

// `keep`: the hash bits kept (all ones; fewer only under the PA_TEST_STR_HASH_BITS collision hook)
__global__ void __launch_bounds__(256) k_str_hash(StrCol c, const uint8_t* valid, int64_t bit_off, int64_t n, uint64_t seed, uint64_t keep, uint64_t* out) {
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (; i < n; i += stride) {
    if (valid && !bit_at(valid, bit_off + i)) { out[i] = 0; continue; }
    const int64_t a = str_off(c, i), b = str_off(c, i + 1);
    out[i] = str_hash64(c.bytes + a, b - a, seed) & keep;
  }
}

__global__ void __launch_bounds__(256) k_str_lengths(StrCol c, const uint32_t* first_row, const uint8_t* key_kind, uint32_t G, uint32_t* len_out) {
  const uint32_t g = blockIdx.x * 256u + threadIdx.x;
  if (g < G) {
    const int64_t r = first_row[g];
    len_out[g] = key_kind[g] == 1 /* KK_NULL */ ? 0u : static_cast<uint32_t>(str_off(c, r + 1) - str_off(c, r));
  }
  if (g == G) len_out[G] = 0;
}

__global__ void __launch_bounds__(256) k_sum_u32(const uint32_t* v, uint32_t n, unsigned long long* out) {
  unsigned long long acc = 0;
  for (uint32_t i = blockIdx.x * 256u + threadIdx.x; i < n; i += gridDim.x * 256u) acc += v[i];
#pragma unroll
  for (int d = 16; d; d >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, d);
  if (lane_id() == 0 && acc) atomicAdd(out, acc);
}

// validity words of unique(): bit g = group g's key is not null (whole words, zero padded)
__global__ void __launch_bounds__(256) k_kind_validity(const uint8_t* key_kind, uint32_t G, uint32_t* out) {
  const uint32_t g = blockIdx.x * 256u + threadIdx.x;
  const bool ok = g < G && key_kind[g] != 1;
  const uint32_t m = __ballot_sync(0xFFFFFFFFu, ok);
  if (lane_id() == 0 && g < (G + 31) / 32 * 32) out[g >> 5] = m;
}

// out_offsets = exclusive scan of the lengths (G + 1 entries); one warp per group copies the bytes
__global__ void __launch_bounds__(256) k_str_gather(StrCol c, const uint32_t* first_row, const uint8_t* key_kind, uint32_t G,
                                                    const uint32_t* out_offsets, uint8_t* out_bytes) {
  const uint32_t g = (blockIdx.x * 256u + threadIdx.x) >> 5;
  if (g >= G || key_kind[g] == 1) return;
  const int64_t r = first_row[g];
  const int64_t a = str_off(c, r);
  const uint32_t len = out_offsets[g + 1] - out_offsets[g];
  for (uint32_t j = lane_id(); j < len; j += 32) out_bytes[out_offsets[g] + j] = c.bytes[a + j];
}

// ---------------------------------------------------------------------------------------------
// utf8 keys across row-range shards.  A record's key word is the seeded hash, so the owner cannot tell two strings
// with one hash apart from the records alone: every exported record carries its group's key bytes — the string at
// the group's first row (global first row - row_base) — in a byte pool next to the records, one uint32 length per
// record, in the order the records were WRITTEN (the scatter places a segment's records by atomics).  The owner maps
// every received record to its merged group, takes the record whose global first row is the group's first row as the
// representative (the first string in row order), and compares every other record's bytes with it.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int64_t str_len(const StrCol& c, int64_t r) { return str_off(c, r + 1) - str_off(c, r); }

// Key bytes per owner of the local groups (before the count gather), like k_partials_count
__global__ void __launch_bounds__(256) k_keystr_count(StrCol c, GroupResult r, uint32_t G, uint32_t nparts, unsigned long long* bytes) {
  __shared__ unsigned long long s_bytes[64];
  if (threadIdx.x < 64) s_bytes[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < G && r.key_kind[g] != KK_NULL) {
    const uint64_t len = static_cast<uint64_t>(str_len(c, r.first_row[g]));
    if (len) atomicAdd(&s_bytes[owner_of(r.key[g], KK_REGULAR, nparts)], static_cast<unsigned long long>(len));
  }
  __syncthreads();
  if (threadIdx.x < nparts && s_bytes[threadIdx.x]) atomicAdd(bytes + threadIdx.x, s_bytes[threadIdx.x]);
}

// The same for the unordered group records of the bucketed path (never a null key)
__global__ void __launch_bounds__(256) k_keystr_count_bk(StrCol c, const BkRec32* recs, uint32_t G, uint32_t nparts, unsigned long long* bytes) {
  __shared__ unsigned long long s_bytes[64];
  if (threadIdx.x < 64) s_bytes[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < G) {
    const uint64_t len = static_cast<uint64_t>(str_len(c, recs[g].first));
    if (len) atomicAdd(&s_bytes[owner_of(recs[g].key, KK_REGULAR, nparts)], static_cast<unsigned long long>(len));
  }
  __syncthreads();
  if (threadIdx.x < nparts && s_bytes[threadIdx.x]) atomicAdd(bytes + threadIdx.x, s_bytes[threadIdx.x]);
}

// One length per exported record (0 for the null key), and the same as 64-bit words for the scan into byte offsets
// (off[n] = 0: after the exclusive scan it is the total)
__global__ void __launch_bounds__(256) k_keystr_lengths(StrCol c, const uint64_t* recs, int words, uint64_t n, int64_t row_base,
                                                        uint32_t* len, unsigned long long* off) {
  const uint64_t i = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x;
  if (i > n) return;
  if (i == n) { off[n] = 0; return; }
  const uint64_t* rec = recs + i * words;
  const bool compact = words == REC_WORDS_COMPACT;
  const uint32_t l = rec_key_null(rec, compact) ? 0u : static_cast<uint32_t>(str_len(c, static_cast<int64_t>(rec_first_row(rec, compact)) - row_base));
  len[i] = l;
  off[i] = l;
}

// One warp per exported record copies its key bytes to out + off[i]
__global__ void __launch_bounds__(256) k_keystr_pack(StrCol c, const uint64_t* recs, int words, uint64_t n, int64_t row_base,
                                                     const unsigned long long* off, uint8_t* out) {
  const uint64_t i = (blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x) >> 5;
  if (i >= n) return;
  const uint64_t len = off[i + 1] - off[i];
  if (!len) return;
  const uint64_t* rec = recs + i * words;
  const int64_t a = str_off(c, static_cast<int64_t>(rec_first_row(rec, words == REC_WORDS_COMPACT)) - row_base);
  uint8_t* dst = out + off[i];
  for (uint64_t j = lane_id(); j < len; j += 32) dst[j] = c.bytes[a + j];
}

// 32-bit lengths -> 64-bit words for the scan into byte offsets (off[n] = 0)
__global__ void __launch_bounds__(256) k_keystr_widen(const uint32_t* len, uint64_t n, unsigned long long* off) {
  const uint64_t i = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x;
  if (i < n) off[i] = len[i];
  else if (i == n) off[n] = 0;
}

constexpr uint32_t KS_COLLISION = 1u, KS_NO_GROUP = 2u;

// Owner side: merged group of every received record; the record that carries the group's global first row becomes
// its representative (exactly one does: a group's first row is one record's first row)
__global__ void __launch_bounds__(256) k_keystr_rep(const uint64_t* recs, int words, uint64_t n, RowIdArgs ids, const uint64_t* first_row_g,
                                                    uint32_t* rec_group, uint32_t* rep, uint32_t* flag) {
  const uint64_t i = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  const uint64_t* rec = recs + i * words;
  const bool compact = words == REC_WORDS_COMPACT;
  const uint32_t g = group_of_key(ids, rec[REC_KEY], rec_key_null(rec, compact));
  rec_group[i] = g;
  if (g >= ids.G) { atomicOr(flag, KS_NO_GROUP); return; }
  if (rec_first_row(rec, compact) == first_row_g[g]) rep[g] = static_cast<uint32_t>(i);
}

// One warp per received record: its key bytes against its group's representative's
__global__ void __launch_bounds__(256) k_keystr_verify(const uint64_t* recs, int words, uint64_t n, const uint32_t* rec_group, const uint32_t* rep,
                                                       const unsigned long long* off, const uint8_t* bytes, uint32_t G, uint32_t* flag) {
  const uint64_t i = (blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x) >> 5;
  if (i >= n) return;
  const uint32_t g = rec_group[i];
  if (g >= G || rec_key_null(recs + i * words, words == REC_WORDS_COMPACT)) return;
  const uint32_t r = rep[g];
  if (r == i) return;
  if (r == 0xFFFFFFFFu) { if (lane_id() == 0) atomicOr(flag, KS_NO_GROUP); return; }
  const uint64_t x = off[i], lx = off[i + 1] - x, y = off[r], ly = off[r + 1] - y;
  bool differ = lx != ly;
  for (uint64_t j = lane_id(); !differ && j < lx; j += 32) differ = bytes[x + j] != bytes[y + j];
  if (__any_sync(0xFFFFFFFFu, differ) && lane_id() == 0) atomicOr(flag, KS_COLLISION);
}

// The merged handle keeps its G representatives only: lengths (off[G] = 0, scanned into offsets) ...
__global__ void __launch_bounds__(256) k_keystr_rep_lengths(const uint32_t* rep, const uint8_t* key_kind, uint32_t G, const unsigned long long* off,
                                                            unsigned long long* out_off, uint32_t* flag) {
  const uint32_t g = blockIdx.x * 256u + threadIdx.x;
  if (g > G) return;
  if (g == G) { out_off[G] = 0; return; }
  const uint32_t r = rep[g];
  if (r == 0xFFFFFFFFu) { atomicOr(flag, KS_NO_GROUP); out_off[g] = 0; return; }
  out_off[g] = key_kind[g] == KK_NULL ? 0ull : off[r + 1] - off[r];
}

// ... and bytes, one warp per group
__global__ void __launch_bounds__(256) k_keystr_rep_gather(const uint32_t* rep, uint32_t G, const unsigned long long* off, const uint8_t* bytes,
                                                           const unsigned long long* out_off, uint8_t* out) {
  const uint32_t g = (blockIdx.x * 256u + threadIdx.x) >> 5;
  if (g >= G) return;
  const uint64_t len = out_off[g + 1] - out_off[g];
  if (!len) return;
  const uint8_t* src = bytes + off[rep[g]];
  for (uint64_t j = lane_id(); j < len; j += 32) out[out_off[g] + j] = src[j];
}

__global__ void __launch_bounds__(256) k_iota_u32(uint32_t* out, uint32_t n) {
  const uint32_t i = blockIdx.x * 256u + threadIdx.x;
  if (i < n) out[i] = i;
}

}  // namespace pa
