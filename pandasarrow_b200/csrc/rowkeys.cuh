// Composite keys that do not pack into 64 bits, or that hold a utf8 column: the key word of a row is a seeded 64-bit
// hash over all its key columns, and the ordinary stages 1-3 group on that 8-byte column, as for a single utf8 key
// (strkeys.cuh).  Exactness comes from the same check: every row against its group's first row (representative).
//   k_row_hash     every row's key columns -> one seeded 64-bit word
//   k_row_verify   every row's null flags and values against its group's representative; also the check of a single
//                  utf8 key (one utf8 column, its validity doubles as the key's null group)
//   k_gather_rep   unique(j): column j at every group's representative, with its null flag
#pragma once
#include "emit.cuh"
#include "strkeys.cuh"

namespace pa {

struct RowKeys {
  const void* col[kMaxKeyCols];      // fixed-width columns: values, already advanced by the array offset
  StrCol str[kMaxKeyCols];           // utf8 / large_utf8 columns
  const uint8_t* valid[kMaxKeyCols]; // validity bitmap (not advanced) or null
  int64_t off[kMaxKeyCols];
  int width[kMaxKeyCols];            // 4 or 8 bytes; 0 = utf8
  int n_cols;
  int64_t n;
};

__device__ __forceinline__ bool rk_null(const RowKeys& k, int j, int64_t i) { return k.valid[j] && !bit_at(k.valid[j], k.off[j] + i); }

__device__ __forceinline__ uint64_t rk_word(const RowKeys& k, int j, int64_t i) {
  return k.width[j] == 8 ? static_cast<const uint64_t*>(k.col[j])[i] : static_cast<uint64_t>(static_cast<const uint32_t*>(k.col[j])[i]);
}

// One step of the row hash: a bijection of x for a fixed h (xor, then the splitmix64 finaliser), so rows that differ in
// one word differ in the word after it
__device__ __forceinline__ uint64_t rk_absorb(uint64_t h, uint64_t x) {
  h ^= x;
  h = (h ^ (h >> 30)) * 0xBF58476D1CE4E5B9ull;
  h = (h ^ (h >> 27)) * 0x94D049BB133111EBull;
  return h ^ (h >> 31);
}

// Column by column: the null flag, then for a valid slot its value bits (a utf8 slot: str_hash64 of its length and
// bytes, seeded with the running hash).  A null slot's value never reaches the hash, as in k_pack_keys.
// `keep`: the hash bits kept (all ones; fewer only under the PA_TEST_STR_HASH_BITS collision hook).
__global__ void __launch_bounds__(256) k_row_hash(RowKeys k, uint64_t seed, uint64_t keep, uint64_t* out) {
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (; i < k.n; i += stride) {
    uint64_t h = seed;
#pragma unroll
    for (int j = 0; j < kMaxKeyCols; ++j) {
      if (j >= k.n_cols) break;
      const bool null = rk_null(k, j, i);
      h = rk_absorb(h, null ? 1u : 2u);
      if (null) continue;
      if (k.width[j]) {
        h = rk_absorb(h, rk_word(k, j, i));
      } else {
        const int64_t a = str_off(k.str[j], i), b = str_off(k.str[j], i + 1);
        h = rk_absorb(h, str_hash64(k.str[j].bytes + a, b - a, h));
      }
    }
    out[i] = h & keep;
  }
}

// Every row against the representative (first row) of the group its hash belongs to; `a` is the read-only
// hash -> group lookup of rowids.cuh built over the hash column.  collision: 1 = two different keys share a hash,
// 2 = a row's hash has no group.
__global__ void __launch_bounds__(256) k_row_verify(RowKeys k, RowIdArgs a, const uint32_t* first_row, uint32_t* collision) {
  int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (; i < a.n; i += stride) {
    const uint32_t g = rowid_lookup(a, i);
    if (g >= a.G) { atomicExch(collision, 2u); continue; }
    const int64_t r = first_row[g];
    if (r == i) continue;
    bool same = true;
#pragma unroll
    for (int j = 0; j < kMaxKeyCols; ++j) {
      if (j >= k.n_cols || !same) break;
      const bool ni = rk_null(k, j, i);
      same = ni == rk_null(k, j, r);
      if (!same || ni) continue;
      if (k.width[j]) {
        same = rk_word(k, j, i) == rk_word(k, j, r);
      } else {
        const StrCol& c = k.str[j];
        const int64_t x = str_off(c, i), lx = str_off(c, i + 1) - x;
        const int64_t y = str_off(c, r), ly = str_off(c, r + 1) - y;
        same = lx == ly;
        for (int64_t b = 0; same && b < lx; ++b) same = c.bytes[x + b] == c.bytes[y + b];
      }
    }
    if (!same) atomicExch(collision, 1u);
  }
}

// Column j at every group's representative row: its null flag as a key kind (KK_NULL / KK_REGULAR, for
// k_kind_validity and unique_strings) and, for a fixed-width column (`col` not null), its value (0 when null)
__global__ void __launch_bounds__(256) k_gather_rep(const void* col, int width, const uint8_t* valid, int64_t off, const uint32_t* first_row,
                                                    uint32_t G, void* out, uint8_t* out_kind) {
  const uint32_t g = blockIdx.x * 256u + threadIdx.x;
  if (g >= G) return;
  const int64_t r = first_row[g];
  const bool null = valid && !bit_at(valid, off + r);
  out_kind[g] = null ? KK_NULL : KK_REGULAR;
  if (!col) return;
  if (width == 8) static_cast<uint64_t*>(out)[g] = null ? 0ull : static_cast<const uint64_t*>(col)[r];
  else static_cast<uint32_t*>(out)[g] = null ? 0u : static_cast<const uint32_t*>(col)[r];
}

}  // namespace pa
