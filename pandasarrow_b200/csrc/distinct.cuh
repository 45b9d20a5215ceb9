// count_distinct per group (GROUPBY_NUMERIC_AGG(count_distinct, int64_t), /root/reference/src/dataframe.cpp:1528;
// arrow::compute "count_distinct" with default CountOptions: distinct NON-NULL values, a memo table keyed by the
// value's bits — so -0.0 / +0.0 and NaNs with different payloads count separately, which is reproduced here).
//
// Exact, sort based:  (group id, widened value bits) of every row  ->  stable radix sort by value, then by id
// (cub::DeviceRadixSort, library code)  ->  one pass counting the positions where (id, bits) changes.
#pragma once
#include "merge.cuh"
#include "rowids.cuh"

namespace pa {

constexpr uint32_t kNoGroup = 0xFFFFFFFFu;

struct DistinctFillArgs {
  RowIdArgs ids;
  const void* vals;
  const uint8_t* vvalid;
  int64_t voff;
  int vw;
  uint64_t* out_bits;
  uint32_t* out_id;      // kNoGroup for null values: sorts behind every real group
};

template <int VC>
__global__ void __launch_bounds__(256) k_distinct_fill(DistinctFillArgs a) {
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (; i < a.ids.n; i += stride) {
    const bool valid = !a.vvalid || bit_at(a.vvalid, a.voff + i);
    a.out_id[i] = valid ? rowid_lookup(a.ids, i) : kNoGroup;
    a.out_bits[i] = valid ? load_wide_rt<VC>(a.vals, i, a.vw) : 0ull;
  }
}

constexpr int CD_PER_THREAD = 8;

// ids ascending (kNoGroup last), bits ascending inside an id.  Every thread walks CD_PER_THREAD consecutive
// positions; the run it ends with (for large groups: its whole chunk) is combined across the warp before the
// one global add per distinct id and warp.
__global__ void __launch_bounds__(256) k_distinct_count(const uint32_t* ids, const uint64_t* bits, int64_t n, unsigned long long* distinct) {
  const int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  const int64_t begin = t * CD_PER_THREAD;
  uint32_t cur = kNoGroup, cnt = 0;
  if (begin < n) {
    uint32_t prev_id = begin ? ids[begin - 1] : kNoGroup;
    uint64_t prev_bits = begin ? bits[begin - 1] : 0ull;
    const bool have_prev = begin > 0;
    for (int j = 0; j < CD_PER_THREAD; ++j) {
      const int64_t i = begin + j;
      if (i >= n) break;
      const uint32_t id = ids[i];
      const uint64_t b = bits[i];
      if (id != cur) {
        if (cur != kNoGroup && cnt) atomicAdd(distinct + cur, static_cast<unsigned long long>(cnt));
        cur = id;
        cnt = 0;
      }
      const bool is_new = !(have_prev || j > 0) || id != prev_id || b != prev_bits;
      if (id != kNoGroup && is_new) ++cnt;
      prev_id = id;
      prev_bits = b;
    }
  }
  const uint32_t peers = __match_any_sync(0xFFFFFFFFu, cur);
  const uint32_t total = __reduce_add_sync(peers, cnt);
  if (cur != kNoGroup && total && static_cast<int>(lane_id()) == __ffs(peers) - 1) atomicAdd(distinct + cur, static_cast<unsigned long long>(total));
}

__global__ void __launch_bounds__(256) k_distinct_emit(const unsigned long long* distinct, uint32_t G, int64_t* out) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < G) out[g] = static_cast<int64_t>(distinct[g]);
}

// ---------------------------------------------------------------------------------------------
// count_distinct across row-range shards.  A per-group count cannot be merged: the same value may occur on several
// shards.  Every shard keeps its distinct (group id, value bits) pairs — the run starts of the sorted arrays above —,
// ships them as (key, bits, flags) to the key's owner (owner_of, like the group records), and the owner inserts
// what it receives into one set of (bits, merged group) and counts the first insertion per group.
// ---------------------------------------------------------------------------------------------

// Run starts of the sorted (id, bits) arrays, without kNoGroup (null values), written to out_id / out_bits in no
// particular order; *cursor ends as the number of distinct pairs.  Same thread -> positions mapping as k_distinct_count.
__global__ void __launch_bounds__(256) k_distinct_pairs(const uint32_t* ids, const uint64_t* bits, int64_t n, uint32_t* out_id,
                                                        uint64_t* out_bits, unsigned long long* cursor) {
  static_assert(CD_PER_THREAD <= 32, "run-start mask");
  const int64_t t = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  const int64_t begin = t * CD_PER_THREAD;
  uint32_t starts = 0;
  if (begin < n) {
    uint32_t prev_id = begin ? ids[begin - 1] : kNoGroup;
    uint64_t prev_bits = begin ? bits[begin - 1] : 0ull;
    for (int j = 0; j < CD_PER_THREAD; ++j) {
      const int64_t i = begin + j;
      if (i >= n) break;
      const uint32_t id = ids[i];
      const uint64_t b = bits[i];
      if (id != kNoGroup && (i == 0 || id != prev_id || b != prev_bits)) starts |= 1u << j;
      prev_id = id;
      prev_bits = b;
    }
  }
  const uint32_t cnt = __popc(starts), lane = lane_id();
  uint32_t incl = cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
    if (lane >= static_cast<uint32_t>(d)) incl += o;
  }
  unsigned long long base = 0;
  if (lane == 31 && incl) base = atomicAdd(cursor, static_cast<unsigned long long>(incl));
  uint64_t pos = __shfl_sync(0xFFFFFFFFu, base, 31) + (incl - cnt);
  for (; starts; starts &= starts - 1, ++pos) {
    const int64_t i = begin + __ffs(starts) - 1;
    out_id[pos] = ids[i];
    out_bits[pos] = bits[i];
  }
}

// Public distinct-pair record (PA_DISTINCT_PAIR_WORDS words): key, value bits (load_wide_rt), flags.
constexpr int DP_KEY = 0, DP_BITS = 1, DP_FLAGS = 2, DP_WORDS = 3;
constexpr uint64_t DPF_KEY_NULL = 1;

struct PairsArgs {
  GroupResult r;               // the handle's groups: key / key kind of every local group id
  const uint32_t* id;          // [n] local group id of pair j
  const uint64_t* bits;        // [n] value bits of pair j
  uint64_t n;
  uint32_t nparts;             // <= 64 (checked by the host)
  unsigned long long* counts;  // [nparts] (k_pairs_count)
  unsigned long long* cursor;  // [nparts] exclusive prefix of the counts (k_pairs_scatter)
  uint64_t* out;               // n * DP_WORDS words, grouped by owner
};

__global__ void __launch_bounds__(256) k_pairs_count(PairsArgs a) {
  __shared__ unsigned int s_cnt[64];
  if (threadIdx.x < 64) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const uint64_t j = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x;
  if (j < a.n) {
    const uint32_t id = a.id[j];
    atomicAdd(&s_cnt[owner_of(a.r.key[id], a.r.key_kind[id], a.nparts)], 1u);
  }
  __syncthreads();
  if (threadIdx.x < a.nparts && s_cnt[threadIdx.x]) atomicAdd(a.counts + threadIdx.x, static_cast<unsigned long long>(s_cnt[threadIdx.x]));
}

// One global cursor add per owner and CTA, as k_partials_scatter.
__global__ void __launch_bounds__(256) k_pairs_scatter(PairsArgs a) {
  __shared__ unsigned int s_cnt[64];
  __shared__ unsigned long long s_base[64];
  if (threadIdx.x < 64) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const uint64_t j = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x;
  uint64_t key = 0;
  uint32_t o = 0, local = 0;
  bool knull = false;
  if (j < a.n) {
    const uint32_t id = a.id[j];
    key = a.r.key[id];
    const uint8_t kind = a.r.key_kind[id];
    knull = kind == KK_NULL;
    o = owner_of(key, kind, a.nparts);
    local = atomicAdd(&s_cnt[o], 1u);
  }
  __syncthreads();
  if (threadIdx.x < a.nparts && s_cnt[threadIdx.x])
    s_base[threadIdx.x] = atomicAdd(a.cursor + threadIdx.x, static_cast<unsigned long long>(s_cnt[threadIdx.x]));
  __syncthreads();
  if (j < a.n) {
    uint64_t* rec = a.out + (s_base[o] + local) * DP_WORDS;
    rec[DP_KEY] = key;
    rec[DP_BITS] = a.bits[j];
    rec[DP_FLAGS] = knull ? DPF_KEY_NULL : 0ull;
  }
}

// Owner side.  Set slot = {value bits, merged group}; empty = all ones, which no pair can be (group ids stay below
// 2^32 - 1).  A slot is claimed with a 128-bit compare-and-swap, and every probe is one: the CAS returns the slot
// as one value, where a plain 16-byte load could see half of a concurrent claim.
struct alignas(16) DistinctSlot {
  unsigned long long bits, g;
};
constexpr int DM_THREADS = 256;
constexpr uint32_t DM_SMEM_GROUPS = 12288;   // per-CTA counters in shared memory (48 KB) up to this many groups

struct DistinctMergeArgs {
  RowIdArgs ids;               // key -> merged group (build_row_lookup over the merged handle's groups)
  const uint64_t* pairs;       // [n * DP_WORDS]
  uint64_t n;
  DistinctSlot* set;           // [cap_mask + 1], filled with all ones
  uint64_t cap_mask;
  unsigned long long* distinct;  // [G] distinct values per merged group
  uint32_t G;
  uint32_t* no_group;          // set to 1 when a pair's key is no merged group
};

// SMEM: G <= DM_SMEM_GROUPS, counts privatised per CTA.  Either way the new insertions of a warp are combined per group
// (__match_any_sync) first: with 1000 groups, many lanes of a warp count for the same one.
template <bool SMEM>
__global__ void __launch_bounds__(DM_THREADS) k_distinct_merge(DistinctMergeArgs a) {
  extern __shared__ unsigned int dm_cnt[];
  if constexpr (SMEM) {
    for (uint32_t g = threadIdx.x; g < a.G; g += DM_THREADS) dm_cnt[g] = 0;
    __syncthreads();
  }
  const uint32_t lane = lane_id();
  const uint64_t stride = static_cast<uint64_t>(gridDim.x) * DM_THREADS;
  // warp-uniform trip count: every lane takes part in __match_any_sync
  for (uint64_t base = blockIdx.x * static_cast<uint64_t>(DM_THREADS) + (threadIdx.x & ~31u); base < a.n; base += stride) {
    const uint64_t i = base + lane;
    uint32_t fresh = kNoGroup;   // merged group whose count this lane's pair raises
    if (i < a.n) {
      const uint64_t* p = a.pairs + i * DP_WORDS;
      const uint64_t b = p[DP_BITS];
      const uint32_t g = group_of_key(a.ids, p[DP_KEY], (p[DP_FLAGS] & DPF_KEY_NULL) != 0);
      if (g == kNoGroup) {
        atomicExch(a.no_group, 1u);
      } else {
        const DistinctSlot empty{~0ull, ~0ull}, mine{b, g};
        uint64_t s = hash_key64(b ^ (static_cast<uint64_t>(g) * 0x9E3779B97F4A7C15ull)) & a.cap_mask;
        for (;;) {
          const DistinctSlot old = atomicCAS(a.set + s, empty, mine);
          if (old.bits == ~0ull && old.g == ~0ull) { fresh = g; break; }
          if (old.bits == b && old.g == g) break;
          s = (s + 1) & a.cap_mask;
        }
      }
    }
    const uint32_t peers = __match_any_sync(0xFFFFFFFFu, fresh);
    if (fresh != kNoGroup && static_cast<int>(lane) == __ffs(peers) - 1) {
      if constexpr (SMEM) atomicAdd(dm_cnt + fresh, static_cast<unsigned int>(__popc(peers)));
      else atomicAdd(a.distinct + fresh, static_cast<unsigned long long>(__popc(peers)));
    }
  }
  if constexpr (SMEM) {
    __syncthreads();
    for (uint32_t g = threadIdx.x; g < a.G; g += DM_THREADS)
      if (dm_cnt[g]) atomicAdd(a.distinct + g, static_cast<unsigned long long>(dm_cnt[g]));
  }
}

}  // namespace pa
