// Group id of every row, ids numbered in first-appearance order — what the reference gets from
// arrow::compute::Grouper::Consume (/root/reference/src/dataframe.cpp:1584).  A second pass over the
// keys against a read-only lookup table built from the finished GroupResult (key -> rank).
#pragma once
#include "gtable.cuh"
#include "resample.cuh"

namespace pa {

struct RowIdArgs {
  // lookup table
  unsigned long long* tkeys;   // [cap]
  uint32_t* tranks;            // [cap]
  uint64_t cap_mask;
  int shift;                   // 64 - log2(cap)
  uint32_t* special;           // [0] rank of the null-key group, [1] rank of the (key == kEmptyKey) group, or 0xFFFFFFFF
  // groups
  const uint64_t* gkey;
  const uint8_t* gkind;
  uint32_t G;
  // rows
  const void* keys;
  const uint8_t* kvalid;
  int64_t koff;
  int kw;
  int64_t n;
  int resample;                // keys are timestamps: the group key is the bucket label
  ResampleSpec rs;
  uint32_t* out;
};

__global__ void __launch_bounds__(256) k_rowid_build(RowIdArgs a) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= a.G) return;
  const uint64_t key = a.gkey[g];
  if (a.gkind[g] == KK_NULL) { a.special[0] = g; return; }
  if (key == kEmptyKey) { a.special[1] = g; return; }
  uint64_t s = gtable_home(key, a.shift);
  for (;;) {
    const uint64_t old = atomicCAS(a.tkeys + s, static_cast<unsigned long long>(kEmptyKey), static_cast<unsigned long long>(key));
    if (old == kEmptyKey) { a.tranks[s] = g; return; }
    s = (s + 1) & a.cap_mask;      // keys are distinct: never equal to `old`
  }
}

// Group id of a (non-null) key value, 0xFFFFFFFF if no group has it.
__device__ __forceinline__ uint32_t key_lookup(const RowIdArgs& a, uint64_t key) {
  if (key == kEmptyKey) return a.special[1];
  uint64_t s = gtable_home(key, a.shift);
  for (;;) {
    const uint64_t k = __ldg(a.tkeys + s);
    if (k == key) return __ldg(a.tranks + s);
    if (k == kEmptyKey) return 0xFFFFFFFFu;
    s = (s + 1) & a.cap_mask;
  }
}

// Group id of a key given by value and null flag instead of by row (merge of distinct pairs, distinct.cuh).
__device__ __forceinline__ uint32_t group_of_key(const RowIdArgs& a, uint64_t key, bool is_null) {
  return is_null ? a.special[0] : key_lookup(a, key);
}

// Group id of row i (0xFFFFFFFF if its key was never aggregated — cannot happen for a finished handle).
__device__ __forceinline__ uint32_t rowid_lookup(const RowIdArgs& a, int64_t i) {
  uint64_t key = load_key_rt(a.keys, i, a.kw);
  if (a.kvalid && !bit_at(a.kvalid, a.koff + i)) return a.special[0];
  if (a.resample) {
    const int64_t tp = static_cast<int64_t>(key) - (a.rs.closed_right ? 1 : 0);
    int64_t lo = 0;
    uint64_t w = 0;
    const int64_t b = rs_locate(a.rs, tp, &lo, &w);
    if (b < 0) return 0xFFFFFFFFu;
    key = static_cast<uint64_t>(rs_label(a.rs, b));
  }
  return key_lookup(a, key);
}

__global__ void __launch_bounds__(256) k_rowid_scan(RowIdArgs a) {
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (; i < a.n; i += stride) a.out[i] = rowid_lookup(a, i);
}

}  // namespace pa
