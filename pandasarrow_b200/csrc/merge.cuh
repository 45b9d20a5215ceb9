// Multi-GPU exchange + merge (SURVEY.md §8e).  Rows are sharded by contiguous range; every GPU
// aggregates its shard (stages 1-3), then
//   1. k_partials_count / k_partials_scatter bucket the local groups by owner = hash(key) % P into
//      fixed-size records, grouped by destination rank (the send buffer of the all-to-all);
//   2. the host exchanges counts and records with an all-to-all over NVLink (NCCL);
//   3. k_merge_insert / k_merge_fold join the received records by key and fold them IN SOURCE-RANK
//      ORDER (at most one record per source and key), so fp64 sums do not depend on arrival order;
//   4. the merged groups are ordered by their global first row.
// Product / variance / stddev travel in a longer record (REC_WORDS_STAGE2): every source ships its two-pass terms
// (M2 = sum of (x - mean)^2 around its own mean, and its product), and k_merge_fold<true> combines them in source-rank
// order with Chan's pairwise update of (n, mean, M2) and a plain product.
// The reference has no multi-device path at all (SURVEY.md §2b); this is new structure.
#pragma once
#include "group_result.cuh"

namespace pa {

// One partial aggregate = PA_REC_WORDS 64-bit words.
constexpr int REC_KEY = 0, REC_FLAGS = 1, REC_SUM = 2, REC_DSUM = 3, REC_COUNT = 4, REC_FIRST_ROW = 5,
              REC_LAST_ROW = 6, REC_MIN = 7, REC_MAX = 8, REC_FIRST_VAL = 9, REC_LAST_VAL = 10, REC_WORDS = 11;
// Stage-2 record (PA_PARTIAL_WORDS_STAGE2): the REC_WORDS words above, then M2 (double bits) and the product (raw 64 bits
// in the value class: double bits for floats, the wrapped (u)int64 otherwise).  RF_HAS_M2 / RF_HAS_PROD say which of the
// two the source's aggregate computed; the mean M2 was taken around is sum / count (floats) or dsum / count (integers),
// the division k_stage2_init does, so the merge recomputes it from the record.
constexpr int REC_M2 = 11, REC_PROD = 12, REC_WORDS_STAGE2 = 13;
constexpr uint64_t RF_KEY_NULL = 1, RF_FIRST_VALID = 2, RF_LAST_VALID = 4, RF_HAS_M2 = 8, RF_HAS_PROD = 16;
// Compact record of the sharded step (pa_groupby_sharded_aggregate) when the aggregate set needs nothing but
// sum / count / first row (sum, mean of floats, count): ONE 32-byte sector per group instead of 88 bytes —
// 100 M groups per rank: 3.2 GB instead of 8.8 GB written, sent and joined.  Internal to the library (both ends of the
// exchange are this code); the public partial record of pa_groupby_partials_export stays PA_PARTIAL_WORDS wide.
constexpr int RC_KEY = 0, RC_SUM = 1, RC_COUNT = 2, RC_FIRST_ROW = 3, REC_WORDS_COMPACT = 4;
constexpr uint64_t RC_KEY_NULL_BIT = 1ull << 63;   // in the count word
__device__ __forceinline__ bool rec_key_null(const uint64_t* rec, bool compact) {
  return compact ? (rec[RC_COUNT] & RC_KEY_NULL_BIT) != 0 : (rec[REC_FLAGS] & RF_KEY_NULL) != 0;
}
__device__ __forceinline__ uint64_t rec_first_row(const uint64_t* rec, bool compact) { return rec[compact ? RC_FIRST_ROW : REC_FIRST_ROW]; }

__device__ __forceinline__ uint32_t owner_of(uint64_t key, uint8_t kind, uint32_t nparts) {
  if (kind == KK_NULL) return 0u;
  return static_cast<uint32_t>(hash_key64(key) % nparts);
}

struct PartialsArgs {
  GroupResult r;
  uint32_t G;
  uint32_t nparts;
  int64_t row_base;            // global row number of local row 0
  // optional first/last values as emitted by k_emit (typed, width vw) + validity bitmaps
  const void* first_vals; const uint32_t* first_valid;
  const void* last_vals; const uint32_t* last_valid;
  int vw;
  bool wide;
  int words;                   // record width: REC_WORDS, REC_WORDS_STAGE2, or REC_WORDS_COMPACT (narrow aggregate sets,
                               // sharded step only)
  const double* m2;            // stage-2 records: per-group M2 / product of the last aggregate, or null when it computed none
  const unsigned long long* prod;
  const uint32_t* G_dev;       // optional: group count on the device (deferred local aggregate)
  const uint32_t* abort_dev;   // optional: non-zero = the local pass failed, send overflow markers
  unsigned long long* counts;  // [nparts] (device)
  unsigned long long* cursor;  // [nparts] running write offsets (device), pre-set to the exclusive prefix of counts
  uint64_t* records;
};

__global__ void __launch_bounds__(256) k_partials_count(PartialsArgs a) {
  __shared__ unsigned int s_cnt[64];
  if (threadIdx.x < 64) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < a.G) atomicAdd(&s_cnt[owner_of(a.r.key[g], a.r.key_kind[g], a.nparts)], 1u);
  __syncthreads();
  if (threadIdx.x < a.nparts && s_cnt[threadIdx.x]) atomicAdd(a.counts + threadIdx.x, static_cast<unsigned long long>(s_cnt[threadIdx.x]));
}

__device__ __forceinline__ uint64_t load_raw(const void* p, uint32_t i, int vw) {
  switch (vw) {
    case 8: return static_cast<const uint64_t*>(p)[i];
    case 4: return static_cast<const uint32_t*>(p)[i];
    case 2: return static_cast<const uint16_t*>(p)[i];
    default: return static_cast<const uint8_t*>(p)[i];
  }
}

__device__ __forceinline__ void write_partial_record(const PartialsArgs& a, uint32_t g, uint8_t kind, uint64_t* rec) {
  if (a.words == REC_WORDS_COMPACT) {   // one sector, two 16-byte stores
    ulonglong2 lo, hi;
    lo.x = a.r.key[g];
    lo.y = a.r.sum[g];
    hi.x = static_cast<uint64_t>(a.r.count[g]) | (kind == KK_NULL ? RC_KEY_NULL_BIT : 0ull);
    hi.y = static_cast<uint64_t>(a.row_base + a.r.first_row[g]);
    reinterpret_cast<ulonglong2*>(rec)[0] = lo;
    reinterpret_cast<ulonglong2*>(rec)[1] = hi;
    return;
  }
  uint64_t flags = kind == KK_NULL ? RF_KEY_NULL : 0;
  rec[REC_KEY] = a.r.key[g];
  rec[REC_SUM] = a.r.sum[g];
  rec[REC_DSUM] = (a.wide && a.r.dsum) ? static_cast<uint64_t>(__double_as_longlong(a.r.dsum[g])) : 0ull;
  rec[REC_COUNT] = a.r.count[g];
  rec[REC_FIRST_ROW] = static_cast<uint64_t>(a.row_base + a.r.first_row[g]);
  rec[REC_LAST_ROW] = a.wide ? static_cast<uint64_t>(a.row_base + a.r.last_row[g]) : 0ull;
  rec[REC_MIN] = a.wide ? a.r.min_ord[g] : kMinInit;
  rec[REC_MAX] = a.wide ? a.r.max_ord[g] : kMaxInit;
  uint64_t fv = 0, lv = 0;
  if (a.first_vals) {
    fv = load_raw(a.first_vals, g, a.vw);
    if (!a.first_valid || ((a.first_valid[g >> 5] >> (g & 31)) & 1u)) flags |= RF_FIRST_VALID;
  }
  if (a.last_vals) {
    lv = load_raw(a.last_vals, g, a.vw);
    if (!a.last_valid || ((a.last_valid[g >> 5] >> (g & 31)) & 1u)) flags |= RF_LAST_VALID;
  }
  rec[REC_FIRST_VAL] = fv;
  rec[REC_LAST_VAL] = lv;
  if (a.words == REC_WORDS_STAGE2) {
    rec[REC_M2] = a.m2 ? static_cast<uint64_t>(__double_as_longlong(a.m2[g])) : 0ull;
    rec[REC_PROD] = a.prod ? a.prod[g] : 0ull;
    flags |= (a.m2 ? RF_HAS_M2 : 0ull) | (a.prod ? RF_HAS_PROD : 0ull);
  }
  rec[REC_FLAGS] = flags;
}

// One global cursor add per owner and CTA (a cursor add per record serialises on nparts addresses:
// 39 ms for 100 M records).  nparts <= 64 (checked by the host, like k_partials_count).
__global__ void __launch_bounds__(256) k_partials_scatter(PartialsArgs a) {
  __shared__ unsigned int s_cnt[64];
  __shared__ unsigned long long s_base[64];
  if (threadIdx.x < 64) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  uint8_t kind = 0;
  uint32_t o = 0, local = 0;
  if (g < a.G) {
    kind = a.r.key_kind[g];
    o = owner_of(a.r.key[g], kind, a.nparts);
    local = atomicAdd(&s_cnt[o], 1u);
  }
  __syncthreads();
  if (threadIdx.x < a.nparts && s_cnt[threadIdx.x])
    s_base[threadIdx.x] = atomicAdd(a.cursor + threadIdx.x, static_cast<unsigned long long>(s_cnt[threadIdx.x]));
  __syncthreads();
  if (g < a.G) write_partial_record(a, g, kind, a.records + (s_base[o] + local) * a.words);
}

// Few groups: no host round trip.  One CTA writes, for every destination rank, a fixed-size block
// of (1 + block_records) records: record 0 is a header (word 0 = number of records that follow, or
// kBlockOverflow when this rank has more groups than a block holds), then the records that rank
// owns.  The blocks are exchanged with an equal-split all-to-all.
constexpr uint64_t kBlockOverflow = ~0ull;
__global__ void __launch_bounds__(1024, 1) k_partials_pack_padded(PartialsArgs a, uint64_t block_records) {
  __shared__ unsigned int s_cnt[64];
  if (threadIdx.x < 64) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const uint64_t stride = (block_records + 1) * REC_WORDS;
  if (a.G_dev) a.G = *a.G_dev;
  const bool overflow = a.G > block_records || (a.abort_dev && *a.abort_dev);
  if (!overflow) {
    for (uint32_t g = threadIdx.x; g < a.G; g += blockDim.x) {
      const uint8_t kind = a.r.key_kind[g];
      const uint32_t o = owner_of(a.r.key[g], kind, a.nparts);
      const uint32_t pos = atomicAdd(&s_cnt[o], 1u);
      write_partial_record(a, g, kind, a.records + o * stride + (1 + pos) * REC_WORDS);
    }
  }
  __syncthreads();
  if (threadIdx.x < a.nparts) {
    uint64_t* hdr = a.records + threadIdx.x * stride;
    hdr[0] = overflow ? kBlockOverflow : static_cast<uint64_t>(s_cnt[threadIdx.x]);
    for (int w = 1; w < REC_WORDS; ++w) hdr[w] = 0;
  }
}

// Received padded blocks (one per source rank) -> contiguous records + the exclusive prefix of the
// per-source counts, both on the device.  One CTA per source.
__global__ void __launch_bounds__(256) k_merge_unpad(const uint64_t* blocks, uint32_t nsrc, uint64_t block_records,
                                                    uint64_t* records, uint64_t* src_offset, uint32_t* status) {
  const uint64_t stride = (block_records + 1) * REC_WORDS;
  const uint32_t s = blockIdx.x;
  uint64_t off = 0, mine = 0;
  bool bad = false;
  for (uint32_t q = 0; q < nsrc; ++q) {
    const uint64_t c = blocks[q * stride];
    if (c == kBlockOverflow || c > block_records) { bad = true; continue; }
    if (q < s) off += c;
    if (q == s) mine = c;
  }
  if (bad) {
    if (threadIdx.x == 0) atomicExch(status + ST_PEER_OVERFLOW, 1u);
    mine = 0;
  }
  if (threadIdx.x == 0) {
    src_offset[s] = bad ? 0 : off;
    if (s == nsrc - 1) src_offset[nsrc] = bad ? 0 : off + mine;
  }
  const uint64_t* src = blocks + s * stride + REC_WORDS;
  uint64_t* dst = records + off * REC_WORDS;
  for (uint64_t w = threadIdx.x; w < mine * REC_WORDS; w += blockDim.x) dst[w] = src[w];
}

struct MergeArgs {
  const uint64_t* records;       // all received records, grouped by source rank
  const uint64_t* src_offset;    // [nsrc + 1] exclusive prefix of the per-source record counts (device)
  uint32_t nsrc;
  int words;                     // record stride: REC_WORDS, REC_WORDS_STAGE2, or REC_WORDS_COMPACT (compact layout, see above)
  uint64_t nrec;                 // upper bound (grid sizing); the exact count is src_offset[nsrc]
  unsigned long long* tkeys;     // cap + 2 keys
  uint64_t cap_mask;
  uint64_t max_probe;            // give up (ST_OVERFLOW) after this many probes: a table sized by a hint may be too small
  uint32_t* idx;                 // [(cap + 2) * nsrc] record index per (slot, source) or 0xFFFFFFFF
  uint32_t* status;
  // compacted, unordered merged groups
  uint64_t* m_first_row;         // sort key
  uint32_t* m_slot;
  // final, ordered
  GroupResult out;
  uint64_t* o_first_val; uint64_t* o_last_val; uint8_t* o_first_valid; uint8_t* o_last_valid;
  uint64_t* o_first_row_g;       // global first row of every merged group
  double* o_m2;                  // stage-2 records: merged M2 / product of every merged group, null when not asked for
  unsigned long long* o_prod;
  const uint32_t* order;         // slot of the r-th merged group (after the sort)
  uint32_t G;
  int vc;
};

__global__ void __launch_bounds__(256) k_merge_insert(MergeArgs a) {
  const uint64_t i = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x;
  if (i >= a.src_offset[a.nsrc]) return;   // (device-side count: padded exchanges do not know it on the host)
  // source rank of record i (nsrc is small: linear scan of the prefix array)
  uint32_t s = 0;
  while (s + 1 < a.nsrc && i >= a.src_offset[s + 1]) ++s;
  const uint64_t* rec = a.records + i * a.words;
  const uint64_t key = rec[REC_KEY];
  const uint64_t cap = a.cap_mask + 1;
  uint64_t slot;
  if (rec_key_null(rec, a.words == REC_WORDS_COMPACT)) slot = cap;
  else if (key == kEmptyKey) slot = cap + 1;
  else {
    // Home slot = TOP bits of the partitioning mix of bucketed.cuh (rp_mix; a different function than owner_of's hash,
    // whose residues the keys of one owner share).  The bucketed path emits its groups bucket after bucket, a bucket is
    // a range of those top bits on every rank, so the records arriving from all sources walk the table front to back
    // together: the slots being filled at any moment are a few MB that stay in L2 instead of 100 M random DRAM sectors.
    // Any other record order just sees one more hash function.
    slot = ((key ^ (key >> 32)) * 0x9E3779B97F4A7C15ull) >> __clzll(static_cast<long long>(a.cap_mask));
    bool done = false;
    for (uint64_t probe = 0; probe < a.max_probe; ++probe) {
      const uint64_t k = __ldcg(a.tkeys + slot);
      if (k == key) { done = true; break; }
      if (k == kEmptyKey) {
        const uint64_t old = atomicCAS(a.tkeys + slot, static_cast<unsigned long long>(kEmptyKey), static_cast<unsigned long long>(key));
        if (old == kEmptyKey || old == key) { done = true; break; }
      }
      slot = (slot + 1) & a.cap_mask;
    }
    if (!done) { atomicExch(a.status + ST_OVERFLOW, 1u); return; }
  }
  a.idx[slot * a.nsrc + s] = static_cast<uint32_t>(i);
}

// One thread per slot: if any source contributed, append (global first row, slot) to the compact list.  One counter
// add per CTA (1024 slots): with one per warp, 100 M groups meant 8 M atomics on a single address — 12 ms.
constexpr int MC_THREADS = 1024;
__global__ void __launch_bounds__(MC_THREADS) k_merge_compact(MergeArgs a) {
  __shared__ uint32_t wcount[MC_THREADS / 32];
  __shared__ uint32_t cta_base;
  const uint64_t nslots = a.cap_mask + 3;
  const uint64_t slot = blockIdx.x * static_cast<uint64_t>(MC_THREADS) + threadIdx.x;
  uint64_t first = ~0ull;
  if (slot < nslots) {
    for (uint32_t s = 0; s < a.nsrc; ++s) {
      const uint32_t i = a.idx[slot * a.nsrc + s];
      if (i == 0xFFFFFFFFu) continue;
      const uint64_t f = rec_first_row(a.records + static_cast<uint64_t>(i) * a.words, a.words == REC_WORDS_COMPACT);
      first = f < first ? f : first;
    }
  }
  const bool occ = first != ~0ull;
  const uint32_t m = __ballot_sync(0xFFFFFFFFu, occ);
  const uint32_t w = threadIdx.x >> 5, lane = lane_id();
  if (lane == 0) wcount[w] = __popc(m);
  __syncthreads();
  if (w == 0) {
    const uint32_t c = wcount[lane];
    uint32_t incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
      if (lane >= static_cast<uint32_t>(d)) incl += o;
    }
    wcount[lane] = incl - c;                      // exclusive prefix of the warps
    if (lane == 31) cta_base = incl ? atomicAdd(a.status + ST_COUNTER, incl) : 0u;
  }
  __syncthreads();
  if (occ) {
    const uint32_t pos = cta_base + wcount[w] + __popc(m & ((1u << lane) - 1u));
    a.m_first_row[pos] = first;
    a.m_slot[pos] = static_cast<uint32_t>(slot);
  }
}

// One thread per merged group (final order): fold the sources in rank order.  STAGE2: REC_WORDS_STAGE2-word records,
// whose M2 and product terms are combined as well — sources without values (count 0) are skipped, the first one that
// has some sets (n, mean, M2), every later one applies Chan's update
//   delta = mean_b - mean, n' = n + n_b, M2 += M2_b + delta^2 n n_b / n', mean += delta n_b / n'
// and the products are multiplied in rank order.  A record without the terms the merge asks for sets ST_NO_TERMS.
template <bool STAGE2>
__global__ void __launch_bounds__(256) k_merge_fold(MergeArgs a) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= a.G) return;
  const uint64_t slot = a.order[g];
  uint64_t key = 0, sum = 0, mn = kMinInit, mx = kMaxInit, cnt = 0, first = ~0ull, last = 0, fv = 0, lv = 0;
  double fsum = 0.0, dsum = 0.0;
  bool knull = false, fvalid = false, lvalid = false, any_last = false;
  uint64_t s2_n = 0;
  double s2_mean = 0.0, s2_m2 = 0.0;
  uint64_t s2_prod = a.vc == VC_F ? static_cast<uint64_t>(__double_as_longlong(1.0)) : 1ull;
  bool s2_missing = false;
  for (uint32_t s = 0; s < a.nsrc; ++s) {
    const uint32_t i = a.idx[slot * a.nsrc + s];
    if (i == 0xFFFFFFFFu) continue;
    if (!STAGE2 && a.words == REC_WORDS_COMPACT) {   // {key, sum, count | null-key bit, global first row}: one 32-byte sector
      const ulonglong2* r2 = reinterpret_cast<const ulonglong2*>(a.records + static_cast<uint64_t>(i) * REC_WORDS_COMPACT);
      const ulonglong2 lo = r2[0], hi = r2[1];
      key = lo.x;
      knull = (hi.x & RC_KEY_NULL_BIT) != 0;
      if (a.vc == VC_F) fsum += __longlong_as_double(static_cast<long long>(lo.y));
      else sum += lo.y;
      cnt += hi.x & ~RC_KEY_NULL_BIT;
      first = hi.y < first ? hi.y : first;
      continue;
    }
    const uint64_t* rec = a.records + static_cast<uint64_t>(i) * (STAGE2 ? REC_WORDS_STAGE2 : REC_WORDS);
    key = rec[REC_KEY];
    const uint64_t flags = rec[REC_FLAGS];
    if constexpr (STAGE2) {
      const uint64_t nb = rec[REC_COUNT];
      if (a.o_m2) {
        if (!(flags & RF_HAS_M2)) s2_missing = true;
        else if (nb) {
          // the mean M2_b was taken around, computed as k_stage2_init computed it
          const double mb = __longlong_as_double(static_cast<long long>(rec[a.vc == VC_F ? REC_SUM : REC_DSUM])) / static_cast<double>(nb);
          const double m2b = __longlong_as_double(static_cast<long long>(rec[REC_M2]));
          if (s2_n == 0) {
            s2_mean = mb;
            s2_m2 = m2b;
          } else {
            const double n = static_cast<double>(s2_n), n_b = static_cast<double>(nb), n2 = static_cast<double>(s2_n + nb);
            const double delta = mb - s2_mean;
            s2_m2 += m2b + delta * delta * n * n_b / n2;
            s2_mean += delta * n_b / n2;
          }
          s2_n += nb;
        }
      }
      if (a.o_prod) {
        if (!(flags & RF_HAS_PROD)) s2_missing = true;
        else if (nb) {
          const uint64_t pb = rec[REC_PROD];
          s2_prod = a.vc == VC_F ? static_cast<uint64_t>(__double_as_longlong(__longlong_as_double(static_cast<long long>(s2_prod)) *
                                                                              __longlong_as_double(static_cast<long long>(pb))))
                                 : s2_prod * pb;   // wraps, like the single-GPU product
        }
      }
    }
    knull = flags & RF_KEY_NULL;
    if (a.vc == VC_F) fsum += __longlong_as_double(static_cast<long long>(rec[REC_SUM]));
    else sum += rec[REC_SUM];
    dsum += __longlong_as_double(static_cast<long long>(rec[REC_DSUM]));
    cnt += rec[REC_COUNT];
    mn = rec[REC_MIN] < mn ? rec[REC_MIN] : mn;
    mx = rec[REC_MAX] > mx ? rec[REC_MAX] : mx;
    if (rec[REC_FIRST_ROW] < first) { first = rec[REC_FIRST_ROW]; fv = rec[REC_FIRST_VAL]; fvalid = flags & RF_FIRST_VALID; }
    if (!any_last || rec[REC_LAST_ROW] >= last) { last = rec[REC_LAST_ROW]; lv = rec[REC_LAST_VAL]; lvalid = flags & RF_LAST_VALID; any_last = true; }
  }
  if (a.vc == VC_F) sum = static_cast<uint64_t>(__double_as_longlong(fsum));
  a.out.key[g] = key;
  a.out.key_kind[g] = knull ? KK_NULL : KK_REGULAR;
  a.out.sum[g] = sum;
  a.out.count[g] = static_cast<uint32_t>(cnt > 0xFFFFFFFFull ? 0xFFFFFFFFull : cnt);
  if (a.out.count64) a.out.count64[g] = cnt;
  a.out.first_row[g] = 0;
  if (!STAGE2 && a.words == REC_WORDS_COMPACT) {   // sum / mean / count only: nobody reads last rows, first / last values or min / max (22 B per group less)
    a.o_first_row_g[g] = first;
    return;
  }
  a.out.last_row[g] = 0;
  if (a.out.min_ord) { a.out.min_ord[g] = mn; a.out.max_ord[g] = mx; }
  if (a.out.dsum) a.out.dsum[g] = dsum;
  a.o_first_row_g[g] = first;
  a.o_first_val[g] = fv;
  a.o_last_val[g] = lv;
  a.o_first_valid[g] = fvalid;
  a.o_last_valid[g] = lvalid;
  if constexpr (STAGE2) {
    if (a.o_m2) a.o_m2[g] = s2_m2;
    if (a.o_prod) a.o_prod[g] = s2_prod;
    if (s2_missing) atomicExch(a.status + ST_NO_TERMS, 1u);
  }
}

// ---------------------------------------------------------------------------------------------
// Few groups (padded exchange): the whole merge in ONE single-CTA kernel — join by key in a
// shared-memory table, fold every key's records in source-rank order, rank the groups by their
// global first row, write the final arrays.  Replaces a chain of ~10 latency-bound launches.
// Limits: <= MS_MAX_REC records in total, <= MS_MAX_GROUPS distinct keys; beyond that the kernel
// sets ST_OVERFLOW and the host runs the general merge.
// ---------------------------------------------------------------------------------------------
constexpr int MS_THREADS = 1024;
constexpr int MS_MAX_REC = 16384;
constexpr int MS_TCAP_LOG2 = 13;
constexpr int MS_TCAP = 1 << MS_TCAP_LOG2;
constexpr int MS_MAX_GROUPS = 4096;
constexpr uint32_t MS_NIL = 0xFFFFu;

struct MergeSmallArgs {
  const uint64_t* blocks;        // received padded blocks, one per source rank
  uint32_t nsrc;
  uint64_t block_records;
  int vc;
  GroupResult out;               // capacity >= min(nsrc * block_records, MS_MAX_GROUPS) + 2
  uint64_t* o_first_val; uint64_t* o_last_val; uint8_t* o_first_valid; uint8_t* o_last_valid;
  uint64_t* o_first_row_g;
  uint32_t* status;              // ST_COUNTER = number of merged groups
};

__global__ void __launch_bounds__(MS_THREADS, 1) k_merge_small(MergeSmallArgs a) {
  extern __shared__ __align__(16) unsigned char ms_smem[];
  unsigned long long* tkeys = reinterpret_cast<unsigned long long*>(ms_smem);      // MS_TCAP + 2 (null / sentinel key)
  unsigned long long* gfirst = tkeys + MS_TCAP + 2;                                 // MS_MAX_GROUPS + 2: global first row of group m
  uint16_t* head = reinterpret_cast<uint16_t*>(gfirst + MS_MAX_GROUPS + 2);         // MS_TCAP + 2: newest record of the slot
  uint16_t* next = head + MS_TCAP + 2;                                              // MS_MAX_REC: older record of the same slot
  uint16_t* gslot = next + MS_MAX_REC;                                              // MS_MAX_GROUPS + 2: slot of group m
  __shared__ uint32_t s_off[65];
  __shared__ uint32_t s_ngroups, s_bad;
  const uint64_t stride = (a.block_records + 1) * REC_WORDS;
  if (threadIdx.x == 0) {
    uint32_t off = 0;
    bool bad = false;
    for (uint32_t s = 0; s < a.nsrc; ++s) {
      const uint64_t c = a.blocks[s * stride];
      s_off[s] = off;
      if (c == kBlockOverflow || c > a.block_records) bad = true;
      else off += static_cast<uint32_t>(c);
    }
    s_off[a.nsrc] = off;
    s_ngroups = 0;
    s_bad = bad ? 1u : (off > MS_MAX_REC ? 2u : 0u);
  }
  for (int i = threadIdx.x; i < MS_TCAP + 2; i += MS_THREADS) { tkeys[i] = kEmptyKey; head[i] = MS_NIL; }
  __syncthreads();
  if (s_bad) {
    if (threadIdx.x == 0) atomicExch(a.status + (s_bad == 1u ? ST_PEER_OVERFLOW : ST_OVERFLOW), 1u);
    return;
  }
  const uint32_t nrec = s_off[a.nsrc];
  auto rec_of = [&](uint32_t i, uint32_t* src) -> const uint64_t* {   // i-th record overall (source-major)
    uint32_t s = 0;
    while (s + 1 < a.nsrc && i >= s_off[s + 1]) ++s;
    *src = s;
    return a.blocks + s * stride + (1 + (i - s_off[s])) * REC_WORDS;
  };
  // phase 1: join by key; every slot keeps a list of its records
  for (uint32_t i = threadIdx.x; i < nrec; i += MS_THREADS) {
    uint32_t src;
    const uint64_t* rec = rec_of(i, &src);
    const uint64_t key = rec[REC_KEY];
    uint32_t slot;
    if (rec[REC_FLAGS] & RF_KEY_NULL) slot = MS_TCAP;
    else if (key == kEmptyKey) slot = MS_TCAP + 1;
    else {
      slot = static_cast<uint32_t>(hash_key64(key ^ 0xA5A5A5A5A5A5A5A5ull)) & (MS_TCAP - 1);
      // Bounded probe: more than MS_MAX_GROUPS distinct keys (skewed ownership) must end in ST_OVERFLOW and the
      // general merge on the host side, never in a full table that threads circle forever.
      bool placed = false;
      for (int probe = 0; probe < MS_TCAP; ++probe) {
        if (*reinterpret_cast<volatile uint32_t*>(&s_ngroups) > MS_MAX_GROUPS) break;
        const uint64_t k = *reinterpret_cast<volatile unsigned long long*>(tkeys + slot);
        if (k == key) { placed = true; break; }
        if (k == kEmptyKey) {
          const uint64_t old = atomicCAS(tkeys + slot, static_cast<unsigned long long>(kEmptyKey), static_cast<unsigned long long>(key));
          if (old == kEmptyKey) {
            if (atomicAdd(&s_ngroups, 1u) >= MS_MAX_GROUPS) atomicExch(a.status + ST_OVERFLOW, 1u);
            placed = true;
            break;
          }
          if (old == key) { placed = true; break; }
        }
        slot = (slot + 1) & (MS_TCAP - 1);
      }
      if (!placed) {   // table (nearly) full: give up on this record, the host reruns the general merge
        atomicExch(a.status + ST_OVERFLOW, 1u);
        continue;
      }
    }
    // push front (16-bit exchange emulated on the containing 32-bit word)
    uint32_t* word = reinterpret_cast<uint32_t*>(head) + (slot >> 1);
    const uint32_t sh = (slot & 1u) * 16u;
    uint32_t old = *reinterpret_cast<volatile uint32_t*>(word), assumed;
    do {
      assumed = old;
      old = atomicCAS(word, assumed, (assumed & ~(0xFFFFu << sh)) | (i << sh));
    } while (old != assumed);
    next[i] = static_cast<uint16_t>((old >> sh) & 0xFFFFu);
  }
  __syncthreads();
  if (*reinterpret_cast<volatile uint32_t*>(a.status + ST_OVERFLOW)) return;
  // phase 2: enumerate the occupied slots; a group's sort key is its smallest global first row
  if (threadIdx.x == 0) s_ngroups = 0;
  __syncthreads();
  for (int slot = threadIdx.x; slot < MS_TCAP + 2; slot += MS_THREADS) {
    uint32_t i = head[slot];
    if (i == MS_NIL) continue;
    uint64_t first = ~0ull;
    for (; i != MS_NIL; i = next[i]) {
      uint32_t src;
      const uint64_t f = rec_of(i, &src)[REC_FIRST_ROW];
      first = f < first ? f : first;
    }
    const uint32_t m = atomicAdd(&s_ngroups, 1u);
    gslot[m] = static_cast<uint16_t>(slot);
    gfirst[m] = first;
  }
  __syncthreads();
  const uint32_t M = s_ngroups;
  // phase 3: rank by first row (distinct: a row belongs to one group), fold in source-rank order, write
  for (uint32_t m = threadIdx.x; m < M; m += MS_THREADS) {
    const uint64_t myf = gfirst[m];
    uint32_t rank = 0;
    for (uint32_t j = 0; j < M; ++j) rank += gfirst[j] < myf;
    const uint32_t slot = gslot[m];
    uint64_t key = 0, sum = 0, mn = kMinInit, mx = kMaxInit, cnt = 0, first = ~0ull, last = 0, fv = 0, lv = 0;
    double fsum = 0.0, dsum = 0.0;
    bool knull = false, fvalid = false, lvalid = false, any_last = false;
    // the list holds at most one record per source; visit the sources in ascending order
    uint32_t done_below = 0;   // sources < done_below are folded
    for (;;) {
      uint32_t best = 0xFFFFFFFFu, best_i = MS_NIL;
      for (uint32_t i = head[slot]; i != MS_NIL; i = next[i]) {
        uint32_t src;
        rec_of(i, &src);
        if (src >= done_below && src < best) { best = src; best_i = i; }
      }
      if (best_i == MS_NIL) break;
      done_below = best + 1;
      uint32_t src;
      const uint64_t* rec = rec_of(best_i, &src);
      key = rec[REC_KEY];
      const uint64_t flags = rec[REC_FLAGS];
      knull = flags & RF_KEY_NULL;
      if (a.vc == VC_F) fsum += __longlong_as_double(static_cast<long long>(rec[REC_SUM]));
      else sum += rec[REC_SUM];
      dsum += __longlong_as_double(static_cast<long long>(rec[REC_DSUM]));
      cnt += rec[REC_COUNT];
      mn = rec[REC_MIN] < mn ? rec[REC_MIN] : mn;
      mx = rec[REC_MAX] > mx ? rec[REC_MAX] : mx;
      if (rec[REC_FIRST_ROW] < first) { first = rec[REC_FIRST_ROW]; fv = rec[REC_FIRST_VAL]; fvalid = flags & RF_FIRST_VALID; }
      if (!any_last || rec[REC_LAST_ROW] >= last) { last = rec[REC_LAST_ROW]; lv = rec[REC_LAST_VAL]; lvalid = flags & RF_LAST_VALID; any_last = true; }
    }
    if (a.vc == VC_F) sum = static_cast<uint64_t>(__double_as_longlong(fsum));
    const uint32_t g = rank;
    a.out.key[g] = key;
    a.out.key_kind[g] = knull ? KK_NULL : KK_REGULAR;
    a.out.sum[g] = sum;
    a.out.count[g] = static_cast<uint32_t>(cnt > 0xFFFFFFFFull ? 0xFFFFFFFFull : cnt);
    if (a.out.count64) a.out.count64[g] = cnt;
    a.out.first_row[g] = 0;
    a.out.last_row[g] = 0;
    if (a.out.min_ord) { a.out.min_ord[g] = mn; a.out.max_ord[g] = mx; }
    if (a.out.dsum) a.out.dsum[g] = dsum;
    a.o_first_row_g[g] = first;
    a.o_first_val[g] = fv;
    a.o_last_val[g] = lv;
    a.o_first_valid[g] = fvalid;
    a.o_last_valid[g] = lvalid;
  }
  if (threadIdx.x == 0) a.status[ST_COUNTER] = M;
}
constexpr size_t MS_SMEM_BYTES = (MS_TCAP + 2) * 8 + (MS_MAX_GROUPS + 2) * 8 + (MS_TCAP + 2) * 2 + MS_MAX_REC * 2 + (MS_MAX_GROUPS + 2) * 2 + 64;

__global__ void __launch_bounds__(256) k_fill_u64(unsigned long long* p, uint64_t n, unsigned long long v) {
  uint64_t i = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x;
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
  for (; i < n; i += stride) p[i] = v;
}

}  // namespace pa
